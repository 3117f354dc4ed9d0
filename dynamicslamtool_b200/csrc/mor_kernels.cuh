// mor_kernels.cuh — the per-frame MOR pipeline as ONE persistent cooperative kernel (sm_100a): crop ground mode,
// clustering, matching, moving tests, tracking and the output cloud. Launched by mor_b200.cu. Every phase cites the
// reference lines (src/MovingObjectRemoval.cpp unless noted) whose behaviour it reproduces; DESIGN.md has the data
// layout and the roofline of each.
//
// Execution model. A frame is a chain of ~12 dependent phases, each a few microseconds of L2-resident work. As
// separate launches every boundary costs ~3 us on B200 plus the ramp and tail of a grid; a barrier between the CTAs of
// one resident grid costs 1.2-1.8 us (profiles/r02_ubench_barrier.txt). So the frame is one kernel, k_frame: a group of
// G CTAs (kT threads each, one CTA per SM) owns one sequence, runs phase after phase over "virtual blocks" (tiles of
// points, cells or clusters, strided over the group: sized from the device-side counts, so no CTA is launched for work
// that does not exist) and meets at a group barrier in between. One sequence takes the whole GPU (G = #SMs); S
// sequences per launch (mor_batch_step_device) take G = #SMs / S CTAs each and run independently side by side.
// The same phase functions can be launched one kernel per phase (k_phase<>, per-phase timing for bench.py), and as
// k_frame_pipe: the front half of one frame (ingest ... cluster selection) on most CTAs beside the back half of the
// frame before it (cluster statistics, transform, match, moving test, chain, filter) on the rest - the throughput mode,
// see the end of the file. Clustering is done on pair lists: an enumerate phase (a warp per cell) and a test phase (a
// thread per light pair, a warp per heavy pair).
#pragma once
#include <cstdio>
#include "mor_device.cuh"
#include "../../include/mor_b200.h"

namespace mor {

constexpr int kT = 1024;         // threads per CTA of the frame kernel: one CTA per SM, up to 64 registers per thread
constexpr int kSingle = kT;      // single-CTA bookkeeping phases use the whole CTA
constexpr int kWarps = kT / 32;
constexpr int kLightPair = 256;  // a cell pair with at most this many point pairs is tested by one thread, a larger one by a warp
constexpr int kLightCnt = 32;    // ... and with at most this many points in either cell (the thread's loop stays short; 7 bits in the packed record)
#ifndef MOR_STAGE_LIGHT  // (a stress build shrinks these to force the overflow paths: -DMOR_STAGE_LIGHT=64 -DMOR_STAGE_HEAVY=16 -DMOR_HARD_CAP=2)
#define MOR_STAGE_LIGHT 3072
#define MOR_STAGE_HEAVY 512
#define MOR_HARD_CAP 96
#endif
constexpr int kStageLight = MOR_STAGE_LIGHT, kStageHeavy = MOR_STAGE_HEAVY;  // pair records a CTA collects in shared memory before they go to the lists (24 + 8 KB)
constexpr size_t kLinkSmem = (size_t)kStageLight * 8 + (size_t)kStageHeavy * 16;
// Clusters per frame that the single-CTA steps take (select: sort keys in shared memory, 128 KB; filter: the removal
// bitset). A frame with more runs the group-wide steps of the large-K path instead (phase_select_large, phase_match_large,
// the LARGE filter).
constexpr int kSmallK = 16384;

enum ErrBits { ERR_CLUSTER_CAP = 1, ERR_MOVING_CAP = 2, ERR_LATTICE_RANGE = 4, ERR_GROUND_CAP = 8, ERR_GRID_RANGE = 16, ERR_EDGE_CAP = 32 };
// counts[] slots in which the filter phase parks its results until filterCloud commits the frame (mor_b200.cu, do_filter)
enum { CNT_SPEC_NOUT = 21, CNT_SPEC_NMO = 22, CNT_SPEC_OVERFLOW = 23 };
// A word after the public counts (never copied out): a pipelined method-1 frame's number of clustering cells, from its
// front half to its back half, which empties the grid after the point-distance search (k_frame_pipe_pde)
enum { CNT_PIPE_CELLS = MOR_NCOUNTS, CNT_ALLOC = MOR_NCOUNTS + 1 };

// One occupied cell of the clustering grid: open-addressing hash table keyed by the packed cell coordinates.
// key == 0 is "empty" (every real key has bit 63 set), so a zeroed table is a clean table.
struct __align__(16) Cell {
    unsigned long long key;
    int start;  // first sorted position of the cell's points (= the cell's union-find node)
    int cnt;
};

struct GridDesc {  // dense grid of the voxel ground modes' ball query (mor_ground.cuh); the clustering grid is sparse
    double ox, oy, oz, inv_h;
    int nx, ny, nz, ncells;
};

struct Scratch {  // all zero between frames: every counter is put back by the frame that used it
    unsigned bar;            // group barrier of k_frame (monotonic within a launch)
    int blocks_done;         // CTAs that have finished the frame
    unsigned bar_back; int blocks_done_back;  // the same for the back group of a pipelined launch (k_frame_pipe)
    unsigned tail_centroids, tail_match_back;
    int n_cells, n_roots, n_light, n_heavy;  // list lengths of the frame
    int n_sorted, pad1;      // bump allocator of the sorted array (phase B)
    unsigned tail_match, tail_chain;  // arrival counters of the phases that end with a single-CTA step
    int ticket_out, out_blocks_done;  // stand-alone filter kernel (repeated filterCloud on one frame)
    int err_early;           // error bits raised before the frame's counts exist
    int n_sel;               // size-valid clusters found by the group-wide select (phase_select_large)
    // voxel ground modes only
    int ticket_ingest, ticket_cells;
    unsigned box_inv_min[3], box_max[3];  // bbox of raw_cloud (ordered keys; mins stored inverted so 0 is neutral)
};

struct TrackState {  // persists across frames (MovingObjectRemoval members, .h:109-128)
    int n_mo[2];      // mo_vec.size(), double-buffered like mo_centroid / mo_conf (see filter phase)
    int res_count, res_head;    // res_vec deque
    int corr_count, corr_head;  // corrs_vec deque
    int frames;
    int extract_overflow;
    int n_markers;    // mo_vec entries the last filterCloud looked up (one bounding-box marker each, cpp:640-642)
};

// Everything a phase needs; one per sequence, read from device memory (P[seq]).
struct FramePtrs {
    // ---- input
    const uint8_t* in; uint32_t n, step, off_x, off_y, off_z, off_i; int in_mode;  // 0: float4 records, 1: aligned fields, 2: byte-assembled
    // ---- config
    float trim_x, trim_y, trim_z, gp_limit, r2, volume_constraint, pde_lb, pde_ub, pde_thr, leave_off, catch_up;
    long long min_cluster, max_cluster;
    int method, opc_factor, moving_confidence, static_confidence;
    int kmax, momax, ring_depth;
    double inv_h, cell_h;      // clustering cell edge h = r/sqrt(3)*(1-2^-10): two points of one cell are always within r
    int skip_ingest;           // voxel ground modes: `cloud` / gp_indices were produced by mor_ground.cuh
    // ---- clustering grid (sparse)
    Cell* table; unsigned table_mask;
    int* cell_list;            // [n_cells] table slot of every occupied cell, in creation order
    unsigned long long* ckey; int* cstart; int* ccnt;  // [n_cells] compact copies: key, first sorted position, points
    int2* pslot;               // [N_c] (table slot, rank inside the cell) of every cloud point
    int* slead;                // [N_c] leader position (cell start = the cell's node) of every sorted position; per frame parity
    // link lists: cell pairs to test (light: one thread, heavy: one warp; compact lists, a CTA adds its records in one
    // block) and the connected pairs found (node A, node B; one segment per CTA of the group, no shared counter)
    int2* light; int light_cap;
    int4* heavy; int heavy_cap;
    int2* edges; int edge_seg; int* edge_cnt;
    int* hook;                 // [N_c, at leader positions] union-find over the nodes: parent word (pointers lead to smaller positions); per frame parity
    int* rsize; int* rmin;     // [N_c, at root positions] per root: points and minimum cloud index (= canonical label) of its component; rmin per frame parity
    int* root_list;            // [n_roots] the roots, in no particular order
    // ---- per-frame scratch
    Scratch* scratch; unsigned long long* st_ingest; unsigned long long* st_out;
    uint8_t* point_class; uint8_t* removed_mask;
    int* cloud_src; float4* gpts; int* gsrc;
    int* label; int* cid_of_root; int* cid_of_pos;  // cluster id by canonical label / by root position (-1: not a size-valid cluster); cid_of_pos per frame parity
    int* scid;                 // cluster id per sorted position
    unsigned long long* acc_sum;  // [kmax*6] hi/lo per axis
    unsigned* acc_box;            // [kmax*6] min xyz, max xyz keys
    unsigned* pacc_box;           // [kmax*6] transformed prev clusters
    float4* tpts;                 // transformed prev cloud points (w = prev cluster id bits, -1 if none)
    float* pct;                   // [kmax*3] transformed prev centroids
    float* pbbox;                 // [kmax*6] decoded
    int* recip_q; int* recip_m; int* match_q; int* match_m; float* match_dist; double* match_score;
    int* match_of_prev; int* mid_of_prev; int* mid_of_cur; double* anchorp; int* newcount;
    unsigned long long* lattice; unsigned lattice_mask;
    uint8_t* cluster_removed; int* found;
    int* marker_cluster;          // [momax] cluster each mo_vec entry was matched to by the last filterCloud
    unsigned long long* phase_ts; // [32] %globaltimer at the start of the frame kernel and after every phase (CTA 0); then the pipelined launch's (TS_FRONT, TS_BACK)
    unsigned long long* cta_trace; // [32][256] debug builds (MOR_CTA_TRACE): when every CTA reached the barrier of every phase
    float4* out;
    // ---- ping-pong frame state: cur / prev
    float4* pts; float4* spts; int* cid; int* cl_root; int* cl_size; float* cl_centroid; uint8_t* cl_flags; float* cl_bbox; int* counts;
    const float4* p_pts; const float4* p_spts; const int* p_cid; const int* p_cl_root; const int* p_cl_size; const float* p_cl_centroid;
    const uint8_t* p_cl_flags; const int* p_counts;
    // ---- persistent tracking state
    TrackState* track; float* mo_centroid; int* mo_conf;
    uint8_t* res_ring; int* res_len; int* corr_ring; int* corr_len;
    Affine12 M; int two_frames;
    int mo_parity;  // which half of the mo_vec double buffer is current
    int pde_ring;   // method 1: search reach in cells, ceil(sqrt(pde_ub)/h)
    int tiles_pts;  // size of the scan status arrays
    int frame_smem; // bytes of dynamic shared memory of the frame kernel
    unsigned lattice_words16;    // lattice size in 16-byte units
    // ---- voxel ground modes only (mor_ground.cuh): dense ball-query grid
    int* cell_count; int* cell_start; int* cell_key; int* skey; GridDesc* dgrid; unsigned long long* st_cells; int tiles_cells; int max_cells;
    // ---- frames with more than kSmallK clusters (handles with kmax > kSmallK only; null otherwise)
    unsigned long long* sort_keys;  // [2 kmax] the select's keys, ping-pong of the merge rounds
    int* nn_cur; float* nn_dist;    // [kmax] per previous cluster: nearest current cluster, its squared distance
    int* nn_prev;                   // [kmax] per current cluster: nearest previous cluster
};

__device__ __forceinline__ unsigned long long global_ns() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
#ifdef MOR_CTA_TRACE  // debug builds: when did this CTA get here? (rows 16.. of the trace are sub-steps of phases; tools/cta_trace.py)
#define MOR_TRACE(row) do { __syncthreads(); if (threadIdx.x == 0 && cta < 256) a.cta_trace[(row) * 256 + cta] = global_ns(); } while (0)
#define MOR_TRACE_NOSYNC(row) do { if (threadIdx.x == 0 && cta < 256) a.cta_trace[(row) * 256 + cta] = global_ns(); } while (0)
#else
#define MOR_TRACE(row)
#define MOR_TRACE_NOSYNC(row)
#endif

// ------------------------------------------------------------------------------------------------ group barrier
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned* p) {
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
// All CTAs of a group (co-resident: cooperative launch) meet here; writes before it are visible after it.
struct GroupBarrier {
    unsigned* ctr; unsigned target, G;
    __device__ __forceinline__ void sync() {
        __syncthreads();
        if (G > 1 && threadIdx.x == 0) {
            target += G;
            // release: the CTA's writes (ordered before this by the barrier above) are visible to whoever acquires the count
            asm volatile("red.release.gpu.global.add.u32 [%0], 1;" ::"l"(ctr) : "memory");
            while (ld_acquire_u32(ctr) < target) {}
        }
        __syncthreads();
    }
};

// The sizes every later phase starts from are final once the ingest phase is over: each CTA reads them once and keeps
// them in shared memory (a phase that fetched them itself would begin with a round trip to L2).
struct FrameVars { int n_cells, nc, ng; };
__device__ __forceinline__ FrameVars& frame_vars() {
    __shared__ FrameVars v;
    return v;
}
template <typename P>
__device__ __forceinline__ void load_frame_vars(const P& a) {
    if (threadIdx.x == 0) {
        FrameVars& v = frame_vars();
        v.n_cells = __ldcg(&a.scratch->n_cells); v.nc = __ldcg(&a.counts[MOR_CNT_NC]); v.ng = __ldcg(&a.counts[MOR_CNT_NG]);
    }
    __syncthreads();
}

// "Last one in does the rest": all CTAs of a group call this when they have finished a phase that a short single-CTA
// step follows; it returns true in the CTA that arrived last, which sees everything the others wrote and runs that
// step right away. The others go on to the next barrier. Against a barrier of its own in front of the single-CTA step
// this saves the barrier's latency and the start-up of a phase. `ctr` counts from zero in every frame.
__device__ __forceinline__ bool group_last_arrival(unsigned* ctr, unsigned G) {
    __shared__ int s_last_in;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned old = 0u;
        if (G > 1) asm volatile("atom.acq_rel.gpu.global.add.u32 %0, [%1], 1;" : "=r"(old) : "l"(ctr) : "memory");
        s_last_in = old == G - 1u;
    }
    __syncthreads();
    return s_last_in != 0;
}

// ------------------------------------------------------------------------------------------------ clustering grid
constexpr int kCellBias = 1 << 20;  // cell coordinates are stored biased, 21 bits per axis
__device__ __forceinline__ unsigned long long cell_pack(int cx, int cy, int cz) {
    return (1ull << 63) | ((unsigned long long)(unsigned)(cz + kCellBias) << 42) | ((unsigned long long)(unsigned)(cy + kCellBias) << 21) |
           (unsigned long long)(unsigned)(cx + kCellBias);
}
__device__ __forceinline__ void cell_unpack(unsigned long long key, int& cx, int& cy, int& cz) {
    cx = (int)(key & 0x1FFFFFull) - kCellBias; cy = (int)((key >> 21) & 0x1FFFFFull) - kCellBias; cz = (int)((key >> 42) & 0x1FFFFFull) - kCellBias;
}
// Cell coordinate of one float coordinate (double arithmetic; identical wherever a point is binned). Range-limited so
// that the +-2 neighbourhood never leaves the 21-bit field; *oob is set for coordinates beyond (|x| > ~2^20 cells).
__device__ __forceinline__ int cell_coord(float v, double inv_h, bool* oob) {
    const double c = floor((double)v * inv_h);
    const double lim = (double)(kCellBias - 8);
    if (c < -lim || c > lim) { *oob = true; return c < 0 ? -(kCellBias - 8) : (kCellBias - 8); }
    return (int)c;
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long* p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ int grid_find_or_insert(const FramePtrs& a, unsigned long long key, bool* created) {
    unsigned slot = hash64(key) & a.table_mask;
    while (true) {  // the CAS is the probe: one round trip whether the cell exists or not
        const unsigned long long old = atomicCAS(&a.table[slot].key, 0ull, key);
        if (old == 0ull) { *created = true; return (int)slot; }
        if (old == key) { *created = false; return (int)slot; }
        slot = (slot + 1) & a.table_mask;
    }
}
// Read-only look-up (the table is complete: after the barrier that follows the insert phase).
__device__ __forceinline__ bool grid_lookup(const FramePtrs& a, unsigned long long key, Cell* out) {
    unsigned slot = hash64(key) & a.table_mask;
    while (true) {
        const uint4 raw = __ldcg(reinterpret_cast<const uint4*>(a.table + slot));
        const unsigned long long cur = ((unsigned long long)raw.y << 32) | raw.x;
        if (cur == key) { out->key = cur; out->start = (int)raw.z; out->cnt = (int)raw.w; return true; }
        if (cur == 0ull) return false;
        slot = (slot + 1) & a.table_mask;
    }
}
// Whole warp: the lanes with `valid` bin their point. Lanes that fall into the same cell (neighbouring beams usually
// do) elect one lane that walks the table and takes one ticket block for the group. Returns (slot, rank in the cell);
// *created is set in the lane that created its cell: the caller enters the new cells into the cell list.
__device__ __forceinline__ int2 grid_insert_warp(const FramePtrs& a, bool valid, unsigned long long key, bool* created) {
    const int lane = threadIdx.x & 31;
    const unsigned grp = __match_any_sync(kFull, valid ? key : (unsigned long long)lane);  // real keys have bit 63 set
    const int leader = __ffs(grp) - 1;
    int slot = 0, base = 0;
    *created = false;
    if (valid && lane == leader) {
        slot = grid_find_or_insert(a, key, created);
        base = atomicAdd(&a.table[slot].cnt, __popc(grp));
    }
    slot = __shfl_sync(kFull, slot, leader);
    base = __shfl_sync(kFull, base, leader);
    return make_int2(slot, base + __popc(grp & ((1u << lane) - 1u)));
}
// Cell-list entries of the cells a warp created, one ticket block of the list per warp.
__device__ __forceinline__ void cell_list_append_warp(const FramePtrs& a, bool created, int slot) {
    const int lane = threadIdx.x & 31;
    const unsigned cmask = __ballot_sync(kFull, created);
    if (!cmask) return;
    int lbase = 0;
    if (lane == __ffs(cmask) - 1) lbase = atomicAdd(&a.scratch->n_cells, __popc(cmask));
    lbase = __shfl_sync(kFull, lbase, __ffs(cmask) - 1);
    if (created) a.cell_list[lbase + __popc(cmask & ((1u << lane) - 1u))] = slot;
}

// ------------------------------------------------------------------------------------------------ octree-leaf lattice
// pcl::octree::OctreePointCloudChangeDetector (cpp:319-330, A13): the leaf lattice of a previous cluster is
// floor((p - anchor)/res) in double, anchored at its first point (PCL 1.8 adoptBoundingBoxToPoint + getKeyBitSize, see
// DESIGN.md); the occupied leaves of every transformed previous cluster go into one global hash set keyed
// (prev cluster, ix, iy, iz).
// A previous frame with more clusters than the 16-bit cluster field holds takes the wide key: 25 bits of cluster (any
// K < 2^25 = the largest max_points) and 13 bits per axis, +-409.6 m around the anchor; beyond either range the frame is
// flagged (ERR_LATTICE_RANGE).
constexpr int kLatticeNarrowK = 65535;
__device__ __forceinline__ bool lattice_key(const double* anchor3, int k, float x, float y, float z, unsigned long long* key, bool wide) {
    const double res = (double)0.1f;
    const long long ix = (long long)floor(((double)x - anchor3[0]) / res);
    const long long iy = (long long)floor(((double)y - anchor3[1]) / res);
    const long long iz = (long long)floor(((double)z - anchor3[2]) / res);
    if (wide) {
        *key = ((unsigned long long)(unsigned)k << 39) | ((unsigned long long)(ix + 4096) << 26) | ((unsigned long long)(iy + 4096) << 13) |
               (unsigned long long)(iz + 4096);
        return ix >= -4096 && ix < 4096 && iy >= -4096 && iy < 4096 && iz >= -4096 && iz < 4096;
    }
    const bool ok = ix >= -32768 && ix < 32768 && iy >= -32768 && iy < 32768 && iz >= -32768 && iz < 32768;
    *key = ((unsigned long long)(unsigned)k << 48) | ((unsigned long long)(ix + 32768) << 32) | ((unsigned long long)(iy + 32768) << 16) |
           (unsigned long long)(iz + 32768);
    return ok;
}

// ===================================================================================== phase A: ingest
// pcl::fromPCLPointCloud2 (cpp:523) + PassThrough x, y (cpp:66-74, A1) + CropBox with removed indices (cpp:78-86, A2),
// fused with the stable two-way partition into `cloud` / gp_indices order (one packed decoupled look-back scan over
// 1024-point tiles) and the binning of every cloud point into the clustering grid.
constexpr int kIngestTile = kT;

__device__ __forceinline__ float load_f32(const uint8_t* p, int mode) {
    if (mode != 2) return __ldg(reinterpret_cast<const float*>(p));
    // records whose stride or field offsets are not multiples of 4 (e.g. the 22-byte velodyne XYZIRT layout)
    const unsigned b0 = __ldg(p), b1 = __ldg(p + 1), b2 = __ldg(p + 2), b3 = __ldg(p + 3);
    return __uint_as_float(b0 | (b1 << 8) | (b2 << 16) | (b3 << 24));
}

__device__ __forceinline__ void frame_housekeeping(const FramePtrs& a, int cta, int G) {
    // work for the two-frame stages that depends on the previous frame only, spread over the group: empty octree-leaf
    // hash set, neutral boxes and lattice anchors of the transformed previous clusters
    if (!a.two_frames) return;
    const uint32_t gtid = (uint32_t)cta * kT + threadIdx.x, stride = (uint32_t)G * kT;
    if (a.method == 2) {
        uint4* lat = reinterpret_cast<uint4*>(a.lattice);
        for (uint32_t t = gtid; t < a.lattice_words16; t += stride) lat[t] = make_uint4(0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu, 0xFFFFFFFFu);
    }
    const uint32_t kp = (uint32_t)a.p_counts[MOR_CNT_K];
    for (uint32_t t = gtid; t < kp * 6u; t += stride) a.pacc_box[t] = (t % 6u) < 3u ? 0xFFFFFFFFu : 0u;
    if (a.method == 2) {
        for (uint32_t t = gtid; t < kp; t += stride) {
            // the first point added to the octree is the previous cluster's first (= minimum cloud index) point, transformed
            const float4 p = a.p_pts[a.p_cl_root[t]];
            const float3 f = xform(a.M, p.x, p.y, p.z);
            const double res = (double)0.1f, eps = (double)1.1920928955078125e-07f;
            const double fv[3] = {(double)f.x, (double)f.y, (double)f.z};
#pragma unroll
            for (int q = 0; q < 3; q++) {
                const double lo = fv[q] - res / 2, hi = fv[q] + res / 2;
                const double side = 2.0 * res - eps;
                const double over = (side - (hi - lo)) / 2.0;
                a.anchorp[t * 3 + q] = lo - over;
            }
        }
    }
}

__device__ __forceinline__ unsigned long long bin_point(const FramePtrs& a, const float4& v, bool* oob) {
    const int cx = cell_coord(v.x, a.inv_h, oob), cy = cell_coord(v.y, a.inv_h, oob), cz = cell_coord(v.z, a.inv_h, oob);
    return cell_pack(cx, cy, cz);
}

__device__ __forceinline__ void phase_ingest(const FramePtrs& a, int cta, int G, bool housekeep = true) {
    if (housekeep) frame_housekeeping(a, cta, G);
    const int ntiles = a.n ? (int)((a.n + kIngestTile - 1) / kIngestTile) : 1;
    __shared__ int s_created, s_cbase;
    // Records that are not plain float4 are read field by field from global memory. The phase is a latency chain, not
    // load-bound: staging the tile in shared memory by one bulk copy was measured slower (profiles/README.md).
    for (int tile = cta; tile < ntiles; tile += G) {
        const uint32_t i = (uint32_t)tile * kIngestTile + threadIdx.x;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        int cls = 0;
        if (threadIdx.x == 0) s_created = 0;
        __syncthreads();  // (also: the previous tile's readers of s_cbase are done)
        if (i < a.n) {
            const uint8_t* p = a.in + (size_t)i * a.step;
            if (a.in_mode == 0) {
                v = __ldg(reinterpret_cast<const float4*>(p));
            } else {
                v.x = load_f32(p + a.off_x, a.in_mode); v.y = load_f32(p + a.off_y, a.in_mode); v.z = load_f32(p + a.off_z, a.in_mode);
                v.w = a.off_i != 0xFFFFFFFFu ? load_f32(p + a.off_i, a.in_mode) : 0.f;
            }
            const bool fin = isfinite(v.x) && isfinite(v.y) && isfinite(v.z);
            const bool in_xy = fin && !(v.x < -a.trim_x || v.x > a.trim_x) && !(v.y < -a.trim_y || v.y > a.trim_y);
            if (in_xy) cls = (v.z < a.gp_limit || v.z > a.trim_z) ? 2 : 1;  // x,y box tests of CropBox are implied by the trim
            a.point_class[i] = (uint8_t)cls;
            a.removed_mask[i] = cls ? 1 : 0;
        }
        // binning first: its table walk overlaps with the scan of the partition below. The new cells of the whole tile take
        // ONE ticket block of the cell list (a ticket per warp would queue some 4000 atomics of a frame on one word)
        bool oob = false, created = false;
        const unsigned long long key = cls == 1 ? bin_point(a, v, &oob) : 0ull;
        const int2 sr = grid_insert_warp(a, cls == 1, key, &created);
        if (oob) atomicOr(&a.scratch->err_early, ERR_GRID_RANGE);
        const unsigned cmask = __ballot_sync(kFull, created);
        int cslot = 0;
        if (cmask) {
            if ((threadIdx.x & 31) == __ffs(cmask) - 1) cslot = atomicAdd(&s_created, __popc(cmask));
            cslot = __shfl_sync(kFull, cslot, __ffs(cmask) - 1) + __popc(cmask & ((1u << (threadIdx.x & 31)) - 1u));
        }
        const unsigned long long packed = (cls == 1 ? 1ull : 0ull) | (cls == 2 ? (1ull << 31) : 0ull);
        unsigned long long total;
        const unsigned long long in_block = block_exclusive_scan<unsigned long long, kT>(packed, &total);  // (barriers: s_created is complete)
        if (threadIdx.x == kT - 1) { const int nc_new = s_created; s_cbase = nc_new ? atomicAdd(&a.scratch->n_cells, nc_new) : 0; }  // its round trip hides behind the prefix
        const unsigned long long before = tile_prefix_wide<kT>(a.st_ingest, tile, total);
        const unsigned long long mine = before + in_block;
        if (created) a.cell_list[s_cbase + cslot] = sr.x;
        if (cls == 1) {
            const int c = (int)(mine & 0x7FFFFFFFull);
            a.pts[c] = v;
            a.cloud_src[c] = (int)i;
            a.pslot[c] = sr;
        } else if (cls == 2) {
            const int gi = (int)((mine >> 31) & 0x7FFFFFFFull);
            a.gpts[gi] = v;
            a.gsrc[gi] = (int)i;
        }
        if (tile == ntiles - 1 && threadIdx.x == 0) {
            const unsigned long long all = before + total;
            const int nc = (int)(all & 0x7FFFFFFFull), ng = (int)((all >> 31) & 0x7FFFFFFFull);
            int* c = a.counts;
            for (int k = 0; k < MOR_NCOUNTS; k++) c[k] = 0;
            c[MOR_CNT_N] = (int)a.n; c[MOR_CNT_NT] = nc + ng; c[MOR_CNT_NC] = nc; c[MOR_CNT_NG] = ng;
            c[MOR_CNT_TWO_FRAMES] = a.two_frames;
            if (a.two_frames) { c[MOR_CNT_KPREV] = a.p_counts[MOR_CNT_K]; c[MOR_CNT_NCPREV] = a.p_counts[MOR_CNT_NC]; }
            c[MOR_CNT_FRAME] = a.track->frames + 1;
            a.track->frames += 1;
        }
    }
}

// Voxel ground modes: `cloud` already exists (k_ground_partition); only the binning is left to do.
__device__ __forceinline__ void phase_bin_cloud(const FramePtrs& a, int cta, int G, bool housekeep = true) {
    if (housekeep) frame_housekeeping(a, cta, G);
    const int nc = a.counts[MOR_CNT_NC];
    for (int base = cta * kT; base < nc; base += G * kT) {
        const int c = base + threadIdx.x;
        bool oob = false;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (c < nc) v = a.pts[c];
        const unsigned long long key = c < nc ? bin_point(a, v, &oob) : 0ull;
        bool created = false;
        const int2 sr = grid_insert_warp(a, c < nc, key, &created);
        cell_list_append_warp(a, created, sr.x);
        if (oob) atomicOr(&a.scratch->err_early, ERR_GRID_RANGE);
        if (c < nc) a.pslot[c] = sr;
    }
}

// Work over [0, n) that needs no CTA-wide cooperation is cut into one contiguous slice per CTA (warp granular): a phase
// is short, so what counts is that all SMs take part, not that a CTA's threads are all busy.
__device__ __forceinline__ void cta_slice(int n, int cta, int G, int* lo, int* hi) {
    const int per = ((n + G - 1) / G + 31) & ~31;
    *lo = min(n, cta * per);
    *hi = min(n, *lo + per);
}

// ===================================================================================== phase B: cell ranges
// Every cell gets its range of the sorted array (its first position = the cell's union-find node) and its compact
// descriptors. The order of the cells in the sorted array is free, so the ranges are handed out by bump allocation -
// 32 cells per warp and atomic - instead of a scan: no tile waits for another, and all CTAs take part.
__device__ __forceinline__ void phase_cells(const FramePtrs& a, int cta, int G) {
    const int lane = threadIdx.x & 31;
    int lo, hi;
    cta_slice(frame_vars().n_cells, cta, G, &lo, &hi);
    for (int base = lo + (threadIdx.x & ~31); base < hi; base += kT) {  // (warp-uniform)
        const int i = base + lane;
        int slot = 0, cnt = 0;
        unsigned long long key = 0ull;
        if (i < hi) {
            slot = a.cell_list[i];
            const uint4 raw = __ldcg(reinterpret_cast<const uint4*>(a.table + slot));
            key = ((unsigned long long)raw.y << 32) | raw.x;
            cnt = (int)raw.w;
        }
        int incl = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(kFull, incl, o); if (lane >= o) incl += t; }
        int wbase = 0;
        if (lane == 31) wbase = atomicAdd(&a.scratch->n_sorted, incl);
        const int start = __shfl_sync(kFull, wbase, 31) + incl - cnt;
        if (i < hi) {
            a.table[slot].start = start;
            a.ckey[i] = key; a.cstart[i] = start; a.ccnt[i] = cnt;
            a.hook[start] = start; a.rsize[start] = 0; a.rmin[start] = 0x7FFFFFFF;
        }
    }
}

__device__ __forceinline__ long long warp_sum_ll(long long v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// Per-cluster accumulation of coordinate sums (optional) and bounding boxes with two levels of aggregation before the
// global atomics: warp (match.any + redux) and block (shared memory). In sorted order a tile of kT consecutive points
// lies inside one cluster most of the time, so a 30k-point cluster costs ~30 sets of atomics instead of 30k. Every
// thread of the block must call.
template <bool WITH_SUMS>
__device__ __forceinline__ void block_cluster_accumulate(unsigned long long* acc_sum, unsigned* acc_box, int k, bool valid, float x, float y, float z) {
    __shared__ int s_k[kWarps];                       // cluster of the warp, -1 = no valid lane, -2 = mixed
    __shared__ unsigned long long s_sum[kWarps][6];
    __shared__ unsigned s_box[kWarps][6];
    __shared__ int s_mode;                            // >= 0: the whole block is cluster s_mode; -1: per-warp
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned vmask = __ballot_sync(kFull, valid);
    const unsigned grp = __match_any_sync(kFull, valid ? k : -1);
    const bool leader = valid && (int)(__ffs(grp) - 1) == lane;
    const bool uniform = vmask != 0 && (grp & vmask) == vmask && valid;  // true in the valid lanes of a one-cluster warp
    const bool warp_uniform = __any_sync(kFull, uniform);
    unsigned bx[6];
    {
        const unsigned kx = fkey(x), ky = fkey(y), kz = fkey(z);
        bx[0] = __reduce_min_sync(grp, kx); bx[1] = __reduce_min_sync(grp, ky); bx[2] = __reduce_min_sync(grp, kz);
        bx[3] = __reduce_max_sync(grp, kx); bx[4] = __reduce_max_sync(grp, ky); bx[5] = __reduce_max_sync(grp, kz);
    }
    unsigned long long sm[6] = {0, 0, 0, 0, 0, 0};
    if (WITH_SUMS) {
        const float v[3] = {x, y, z};
#pragma unroll
        for (int q = 0; q < 3; q++) {
            long long h, l;
            split_fixed(v[q], h, l);  // h in [-2^31, 2^31), l in [0, 2^30): summed in 16/15-bit pieces so redux.add (32-bit) cannot overflow
            const long long sh = ((long long)__reduce_add_sync(grp, (int)(h >> 16)) << 16) + (long long)__reduce_add_sync(grp, (int)(h & 0xFFFF));
            const long long sl = ((long long)__reduce_add_sync(grp, (int)(l >> 15)) << 15) + (long long)__reduce_add_sync(grp, (int)(l & 0x7FFF));
            sm[q * 2] = (unsigned long long)sh; sm[q * 2 + 1] = (unsigned long long)sl;
        }
    }
    __syncthreads();  // the previous tile's readers of s_k / s_sum / s_box are done
    if (warp_uniform && leader) {
#pragma unroll
        for (int q = 0; q < 6; q++) { s_box[warp][q] = bx[q]; if (WITH_SUMS) s_sum[warp][q] = sm[q]; }
    }
    const int k_first = __shfl_sync(kFull, k, vmask ? __ffs(vmask) - 1 : 0);
    if (lane == 0) s_k[warp] = !vmask ? -1 : (warp_uniform ? k_first : -2);
    __syncthreads();
    if (warp == 0) {
        const int wk = lane < kWarps ? s_k[lane] : -1;
        const unsigned has = __ballot_sync(kFull, wk != -1);
        const int first = has ? __shfl_sync(kFull, wk, __ffs(has) - 1) : -1;
        const bool same = __all_sync(kFull, wk == -1 || (wk == first && wk >= 0));
        if (lane == 0) s_mode = (has && same) ? first : -1;
    }
    __syncthreads();
    const int mode = s_mode;
    if (mode >= 0) {  // the whole block is one cluster: one set of atomics
        if (threadIdx.x < 6) {
            unsigned v = threadIdx.x < 3 ? 0xFFFFFFFFu : 0u;
            for (int w = 0; w < kWarps; w++)
                if (s_k[w] >= 0) v = threadIdx.x < 3 ? min(v, s_box[w][threadIdx.x]) : max(v, s_box[w][threadIdx.x]);
            if (threadIdx.x < 3) atomicMin(acc_box + mode * 6 + threadIdx.x, v); else atomicMax(acc_box + mode * 6 + threadIdx.x, v);
        } else if (WITH_SUMS && threadIdx.x >= 32 && threadIdx.x < 38) {
            const int q = threadIdx.x - 32;
            unsigned long long v = 0;
            for (int w = 0; w < kWarps; w++)
                if (s_k[w] >= 0) v += s_sum[w][q];
            atomicAdd(acc_sum + mode * 6 + q, v);
        }
    } else if (leader) {  // one set of atomics per (warp, cluster) group
        unsigned* b = acc_box + k * 6;
        atomicMin(b + 0, bx[0]); atomicMin(b + 1, bx[1]); atomicMin(b + 2, bx[2]);
        atomicMax(b + 3, bx[3]); atomicMax(b + 4, bx[4]); atomicMax(b + 5, bx[5]);
        if (WITH_SUMS) {
#pragma unroll
            for (int q = 0; q < 6; q++) atomicAdd(acc_sum + k * 6 + q, sm[q]);
        }
    }
}

// pcl_ros::transformPointCloud of every previous-frame cluster (cpp:544-551, A12), the bounding box of the transformed
// points (getMinMax3D runs after the transform, cpp:272) and, for method 2, their octree leaves (cpp:319-324). Depends
// on the previous frame only: it runs beside the single-CTA cluster selection, on the CTAs that one does not need.
// One point's work in steps that each end at a dependent load (load, look-up, finish), so that the pipelined back half
// can run it beside the cluster statistics with both chains of loads in flight at once (stats_transform).
struct XformItem { float4 p; int k; float3 t; };
__device__ __forceinline__ void xform_load(const FramePtrs& a, int s, int hi, XformItem& it) {
    it.k = -1; it.t = make_float3(0, 0, 0);
    if (s < hi) it.p = a.p_spts[s];
}
__device__ __forceinline__ void xform_lookup(const FramePtrs& a, int s, int hi, XformItem& it) {
    if (s < hi) it.k = a.p_cid[__float_as_int(it.p.w)];
}
__device__ __forceinline__ void xform_finish(const FramePtrs& a, int s, int hi, bool wide, XformItem& it) {
    if (s >= hi) return;
    const int c = __float_as_int(it.p.w), k = it.k;
    if (k >= 0) {
        it.t = xform(a.M, it.p.x, it.p.y, it.p.z);
        a.tpts[c] = make_float4(it.t.x, it.t.y, it.t.z, __int_as_float(k));
        if (a.method == 2) {
            unsigned long long key;
            if (lattice_key(a.anchorp + (size_t)k * 3, k, it.t.x, it.t.y, it.t.z, &key, wide)) hset_insert(a.lattice, a.lattice_mask, key);
            else atomicOr(&a.scratch->err_early, ERR_LATTICE_RANGE);
        }
    } else {
        a.tpts[c] = make_float4(0, 0, 0, __int_as_float(-1));
    }
}
template <bool LK>
__device__ __forceinline__ bool lattice_wide(const FramePtrs& a) { return LK && a.p_counts[MOR_CNT_K] > kLatticeNarrowK; }
template <bool LK>
__device__ __forceinline__ void transform_range(const FramePtrs& a, int lo, int hi) {
    const bool wide = lattice_wide<LK>(a);
    for (int base = lo; base < hi; base += kT) {
        const int s = base + threadIdx.x;
        XformItem it;
        xform_load(a, s, hi, it);
        xform_lookup(a, s, hi, it);
        xform_finish(a, s, hi, wide, it);
        block_cluster_accumulate<false>(nullptr, a.pacc_box, it.k, it.k >= 0, it.t.x, it.t.y, it.t.z);
    }
}
template <bool LK>
__device__ __forceinline__ void phase_transform(const FramePtrs& a, int cta, int G) {
    if (!a.two_frames || (G > 1 && cta == 0)) return;  // CTA 0 selects the clusters meanwhile
    int lo, hi;
    cta_slice(a.p_counts[MOR_CNT_NC], G > 1 ? cta - 1 : 0, G > 1 ? G - 1 : 1, &lo, &hi);
    transform_range<LK>(a, lo, hi);
}


// ===================================================================================== phase C: scatter
// Cloud points into cell order (float4 xyz + cloud index): slot = cell start + the rank taken at binning time.
__device__ __forceinline__ void phase_scatter(const FramePtrs& a, int cta, int G) {
    int lo, hi;
    cta_slice(frame_vars().nc, cta, G, &lo, &hi);
    for (int c = lo + threadIdx.x; c < hi; c += kT) {
        const int2 sr = a.pslot[c];
        const int start = __ldcg(&a.table[sr.x].start);
        float4 p = a.pts[c];
        p.w = __int_as_float(c);
        a.spts[start + sr.y] = p;
        a.slead[start + sr.y] = start;
        atomicMin(&a.rmin[start], c);  // the cell's minimum cloud index: its component's canonical label is the minimum over its cells
    }
}

// ===================================================================================== phase D: link
// pcl::EuclideanClusterExtraction's radius graph (cpp:213-218; A5-A7) on cell granularity. Any two points of one cell
// are neighbours (cell diagonal < r), so a cell is one node (named by the first sorted position of its points), and a
// neighbour lies at most 2 cells away per axis: cell A must be tested against the 62 cells of its 5x5x5 block that
// precede it in (dz,dy,dx) order (the other 62 test A from their side). Two cells are connected iff some point pair has
// L2_Simple distance < r2 (strict).
//
// D1, enumerate: one warp per cell; lane l looks up neighbours l and l+32 in the hash table, both probes in flight
// together. Every occupied neighbour becomes one record of the group's pair lists (per-CTA segments, no shared
// counter): a LIGHT pair (at most kLightPair point pairs) or a HEAVY pair. The warp also leaves the cell's minimum
// cloud index and, for crowded cells, its tight bounding box.
// D2, test: the lists are dealt out evenly over the whole group. A light pair takes one THREAD (a few dozen distance
// tests with early exit; ~60k pairs keep every thread of the GPU busy for one pass), a heavy pair one WARP: a probe of
// samples first (a heavy pair is nearly always connected and nearly any sample shows it), bounding-box pruning and the
// full scan only when the probe finds nothing. Connected pairs are RECORDED (edges, per-CTA segments) and the larger
// node of a pair is pointed at the smaller one (atomicMin on its own word): the forest phase E starts from.
// The frame kernel is 220-290 KB of code, more than an SM's instruction cache holds, yet keeping the large once-per-frame
// steps out of line was measured slower (8.6k vs 9.0k frames/s on C2, profiles/README.md): they are inlined.
#ifdef MOR_DEBUG_BOUNDS
#define MOR_CHECK(cond, tag, v) do { if (!(cond)) { printf("BOUNDS %s: %d (line %d, cta %d thread %d)\n", tag, (int)(v), __LINE__, (int)blockIdx.x, (int)threadIdx.x); } } while (0)
#else
#define MOR_CHECK(cond, tag, v)
#endif
struct BoxF { float lx, ly, lz, hx, hy, hz; };
// Tight bounding box of the n points from sorted position `start`, by the whole warp (only the few heavy pairs whose
// probe found nothing need boxes, so they are made on demand).
__device__ __forceinline__ BoxF warp_box(const FramePtrs& a, int start, int n, int lane) {
    unsigned mnx = 0xFFFFFFFFu, mny = 0xFFFFFFFFu, mnz = 0xFFFFFFFFu, mxx = 0u, mxy = 0u, mxz = 0u;
    for (int k = lane; k < n; k += 32) {
        const float4 p = a.spts[start + k];
        const unsigned kx = fkey(p.x), ky = fkey(p.y), kz = fkey(p.z);
        mnx = min(mnx, kx); mny = min(mny, ky); mnz = min(mnz, kz); mxx = max(mxx, kx); mxy = max(mxy, ky); mxz = max(mxz, kz);
    }
    BoxF b;
    b.lx = fkey_inv(__reduce_min_sync(kFull, mnx)); b.ly = fkey_inv(__reduce_min_sync(kFull, mny)); b.lz = fkey_inv(__reduce_min_sync(kFull, mnz));
    b.hx = fkey_inv(__reduce_max_sync(kFull, mxx)); b.hy = fkey_inv(__reduce_max_sync(kFull, mxy)); b.hz = fkey_inv(__reduce_max_sync(kFull, mxz));
    return b;
}
// conservative squared distance from a point to a box: no point of the box can be closer
__device__ __forceinline__ float box_point_d2(const BoxF& b, float x, float y, float z) {
    const float ex = fmaxf(fmaxf(b.lx - x, x - b.hx), 0.f), ey = fmaxf(fmaxf(b.ly - y, y - b.hy), 0.f), ez = fmaxf(fmaxf(b.lz - z, z - b.hz), 0.f);
    return ex * ex + ey * ey + ez * ez;
}
__device__ __forceinline__ float box_box_d2(const BoxF& p, const BoxF& q) {
    const float ex = fmaxf(fmaxf(p.lx - q.hx, q.lx - p.hx), 0.f), ey = fmaxf(fmaxf(p.ly - q.hy, q.ly - p.hy), 0.f), ez = fmaxf(fmaxf(p.lz - q.hz, q.lz - p.hz), 0.f);
    return ex * ex + ey * ey + ez * ez;
}

// Whole warp on one heavy cell pair (A: cntA points from sorted position sA, B: cB points from sB): is there a point
// pair within r? Three steps of growing cost.
// (1) Probe: 32 samples of B (one per lane) against up to 32 samples of A, spread over the cells, a vote after every
// sample of A. In LiDAR data a crowded cell is connected to every crowded cell around it, and the first or second
// sample shows it (C2: 6400 of 6470 connected heavy pairs per frame).
__device__ __forceinline__ bool heavy_probe(const float4& qa, const float4& qb, float r2) {  // the lane's sample of A and of B
    for (int t = 0; t < 32; t++) {
        const int u = (int)(__brev((unsigned)t) >> 27);  // 0, 16, 8, 24, ...: far apart first
        const float ax = __shfl_sync(kFull, qa.x, u), ay = __shfl_sync(kFull, qa.y, u), az = __shfl_sync(kFull, qa.z, u);
        if (__any_sync(kFull, sqdist3(ax, ay, az, qb.x, qb.y, qb.z) < r2)) return true;
    }
    return false;
}
// (2) The cells' bounding boxes: most unconnected pairs end here.
struct HeavyBoxes { BoxF A, B; };
__device__ __forceinline__ bool heavy_boxes_apart(const FramePtrs& a, int sA, int cntA, int sB, int cB, HeavyBoxes* hb, int lane) {
    hb->A = warp_box(a, sA, cntA, lane);
    hb->B = warp_box(a, sB, cB, lane);
    return box_box_d2(hb->A, hb->B) > a.r2 * 1.00001f;
}
// (3) Full scan of one chunk of 32 points of B (from b0) against all of A, both pruned by the other cell's box: A in
// blocks of 32 per coalesced load, four blocks in flight, every candidate point broadcast by shuffle to all lanes.
__device__ __forceinline__ bool heavy_scan_chunk(const FramePtrs& a, const HeavyBoxes& hb, int sA, int cntA, int sB, int cB, int b0, int lane) {
    const float r2 = a.r2, r2_prune = a.r2 * 1.00001f;
    const float4* A = a.spts + sA;
    const int b = b0 + lane;
    bool valid = b < cB;
    float4 pb = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid) pb = a.spts[sB + b];
    float4 pa[4];
#pragma unroll
    for (int q = 0; q < 4; q++) pa[q] = A[min(32 * q + lane, cntA - 1)];  // (in flight together with B's points)
    if (valid) valid = box_point_d2(hb.A, pb.x, pb.y, pb.z) <= r2_prune;
    if (!__any_sync(kFull, valid)) return false;
    for (int a0 = 0; a0 < cntA; a0 += 128) {
        if (a0) {
#pragma unroll
            for (int q = 0; q < 4; q++) pa[q] = A[min(a0 + 32 * q + lane, cntA - 1)];
        }
        bool h = false;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const bool av = a0 + 32 * q + lane < cntA && box_point_d2(hb.B, pa[q].x, pa[q].y, pa[q].z) <= r2_prune;
            for (unsigned m = __ballot_sync(kFull, av); m; m &= m - 1) {
                const int u = __ffs(m) - 1;
                const float ax = __shfl_sync(kFull, pa[q].x, u), ay = __shfl_sync(kFull, pa[q].y, u), az = __shfl_sync(kFull, pa[q].z, u);
                h |= sqdist3(ax, ay, az, pb.x, pb.y, pb.z) < r2;
            }
        }
        if (__any_sync(kFull, h && valid)) return true;
    }
    return false;
}

// Both neighbours of a lane are looked up with their first probes in flight together.
__device__ __forceinline__ void grid_lookup2(const FramePtrs& a, bool v0, unsigned long long k0, bool v1, unsigned long long k1, int2* sc0, int2* sc1) {
    unsigned s0 = hash64(k0) & a.table_mask, s1 = hash64(k1) & a.table_mask;
    uint4 r0 = make_uint4(0u, 0u, 0u, 0u), r1 = r0;
    if (v0) r0 = __ldcg(reinterpret_cast<const uint4*>(a.table + s0));
    if (v1) r1 = __ldcg(reinterpret_cast<const uint4*>(a.table + s1));
    *sc0 = make_int2(0, 0); *sc1 = make_int2(0, 0);
    while (v0) {
        const unsigned long long cur = ((unsigned long long)r0.y << 32) | r0.x;
        if (cur == k0) { *sc0 = make_int2((int)r0.z, (int)r0.w); break; }
        if (cur == 0ull) break;
        s0 = (s0 + 1) & a.table_mask;
        r0 = __ldcg(reinterpret_cast<const uint4*>(a.table + s0));
    }
    while (v1) {
        const unsigned long long cur = ((unsigned long long)r1.y << 32) | r1.x;
        if (cur == k1) { *sc1 = make_int2((int)r1.z, (int)r1.w); break; }
        if (cur == 0ull) break;
        s1 = (s1 + 1) & a.table_mask;
        r1 = __ldcg(reinterpret_cast<const uint4*>(a.table + s1));
    }
}

struct LinkShared { int n_light, n_heavy, g_light, g_heavy; };

// The lanes with f0 / f1 add one record each: to the CTA's staging area in shared memory, or - once that is full -
// straight to the list.
template <typename T>
__device__ __forceinline__ void stage_append2(const FramePtrs& a, T* stage, int stage_cap, int* s_count, T* list, int list_cap, int* g_count,
                                              bool f0, bool f1, const T& v0, const T& v1, int lane) {
    const unsigned m0 = __ballot_sync(kFull, f0), m1 = __ballot_sync(kFull, f1);
    if (!(m0 | m1)) return;
    int base = 0;
    if (lane == 0) base = atomicAdd(s_count, __popc(m0) + __popc(m1));
    base = __shfl_sync(kFull, base, 0);
    const int w0 = base + __popc(m0 & ((1u << lane) - 1u)), w1 = base + __popc(m0) + __popc(m1 & ((1u << lane) - 1u));
#pragma unroll
    for (int q = 0; q < 2; q++) {
        const bool f = q ? f1 : f0;
        const int w = q ? w1 : w0;
        if (!f) continue;
        if (w < stage_cap) { stage[w] = q ? v1 : v0; continue; }
        const int g = atomicAdd(g_count, 1);
        if (g < list_cap) list[g] = q ? v1 : v0; else atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_EDGE_CAP);
    }
}

// light record: (start | (count - 1) << 25) of both cells; heavy record: (start A, count A, start B, count B)
__device__ __forceinline__ void enumerate_cell(const FramePtrs& a, int i, LinkShared& ls, int2* s_light, int4* s_heavy, int lane) {
    const unsigned long long key = a.ckey[i];
    const int startA = a.cstart[i], cntA = a.ccnt[i];
    MOR_CHECK(startA >= 0 && cntA > 0 && startA + cntA <= a.counts[MOR_CNT_NC], "cellA", cntA);
    int cx, cy, cz;
    cell_unpack(key, cx, cy, cz);
    // the 62 preceding cells of the 5x5x5 block: offset index n = (dz+2)*25 + (dy+2)*5 + (dx+2) < 62
    int2 nb[2];  // (start, cnt) of the lane's two neighbour cells, cnt 0 = empty
    {
        const int n0 = lane, n1 = lane + 32;
        const unsigned long long k0 = cell_pack(cx + n0 % 5 - 2, cy + (n0 / 5) % 5 - 2, cz + n0 / 25 - 2);
        const unsigned long long k1 = cell_pack(cx + n1 % 5 - 2, cy + (n1 / 5) % 5 - 2, cz + n1 / 25 - 2);
        grid_lookup2(a, true, k0, n1 < 62, k1, &nb[0], &nb[1]);
        MOR_CHECK(nb[0].y >= 0 && nb[0].x >= 0 && nb[0].x + nb[0].y <= a.counts[MOR_CNT_NC], "nb0", nb[0].y);
        MOR_CHECK(nb[1].y >= 0 && nb[1].x >= 0 && nb[1].x + nb[1].y <= a.counts[MOR_CNT_NC], "nb1", nb[1].y);
    }
    bool light[2], heavy[2];
#pragma unroll
    for (int q = 0; q < 2; q++) {
        const bool occ = nb[q].y > 0;
        light[q] = occ && cntA <= kLightCnt && nb[q].y <= kLightCnt && cntA * nb[q].y <= kLightPair;
        heavy[q] = occ && !light[q];
    }
    const int wa = startA | ((cntA - 1) << 25);
    stage_append2<int2>(a, s_light, kStageLight, &ls.n_light, a.light, a.light_cap, &a.scratch->n_light, light[0], light[1],
                        make_int2(wa, nb[0].x | ((nb[0].y - 1) << 25)), make_int2(wa, nb[1].x | ((nb[1].y - 1) << 25)), lane);
    stage_append2<int4>(a, s_heavy, kStageHeavy, &ls.n_heavy, a.heavy, a.heavy_cap, &a.scratch->n_heavy, heavy[0], heavy[1],
                        make_int4(startA, cntA, nb[0].x, nb[0].y), make_int4(startA, cntA, nb[1].x, nb[1].y), lane);
}

__device__ __forceinline__ void phase_link(const FramePtrs& a, int cta, int G, unsigned long long* dyn) {
    __shared__ LinkShared ls;
    int2* s_light = reinterpret_cast<int2*>(dyn);
    int4* s_heavy = reinterpret_cast<int4*>(dyn + kStageLight);
    const int n_cells = frame_vars().n_cells;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (threadIdx.x == 0) { ls.n_light = 0; ls.n_heavy = 0; a.edge_cnt[cta] = 0; }
    __syncthreads();
    phase_scatter(a, cta, G);  // independent of the enumeration: both need the cell ranges only
    // an equal share of the cells for every CTA, a warp per cell (from the last warp down: the first warps hold the scatter)
    const int per = (n_cells + G - 1) / G, lo = min(n_cells, cta * per), hi = min(n_cells, lo + per);
    for (int i = lo + (kWarps - 1 - warp); i < hi; i += kWarps) enumerate_cell(a, i, ls, s_light, s_heavy, lane);
    __syncthreads();
    // the CTA's records go to the lists in one block each: one atomic per CTA and list
    const int nl = min(ls.n_light, kStageLight), nh = min(ls.n_heavy, kStageHeavy);
    if (threadIdx.x == 0 && nl) ls.g_light = atomicAdd(&a.scratch->n_light, nl);
    if (threadIdx.x == 32 && nh) ls.g_heavy = atomicAdd(&a.scratch->n_heavy, nh);
    __syncthreads();
    for (int t = threadIdx.x; t < nl; t += kT) {
        const int g = ls.g_light + t;
        if (g < a.light_cap) a.light[g] = s_light[t]; else atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_EDGE_CAP);
    }
    for (int t = threadIdx.x; t < nh; t += kT) {
        const int g = ls.g_heavy + t;
        if (g < a.heavy_cap) a.heavy[g] = s_heavy[t]; else atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_EDGE_CAP);
    }
}

template <int BLK>
__device__ __forceinline__ bool light_pair_connected(const float4* S, int cS, const float4* L, int cL, float r2) {
    for (int k0 = 0; k0 < cS; k0 += BLK) {
        float sx[BLK], sy[BLK], sz[BLK];
#pragma unroll
        for (int q = 0; q < BLK; q++) { const float4 p = S[min(k0 + q, cS - 1)]; sx[q] = p.x; sy[q] = p.y; sz[q] = p.z; }  // (the last block may repeat a point)
        // the block's bounding box: a point of L farther than r from it needs no test against the block (two thirds of the
        // tests belong to unconnected pairs, whose points mostly lie well apart)
        BoxF bx = {sx[0], sy[0], sz[0], sx[0], sy[0], sz[0]};
#pragma unroll
        for (int q = 1; q < BLK; q++) {
            bx.lx = fminf(bx.lx, sx[q]); bx.ly = fminf(bx.ly, sy[q]); bx.lz = fminf(bx.lz, sz[q]);
            bx.hx = fmaxf(bx.hx, sx[q]); bx.hy = fmaxf(bx.hy, sy[q]); bx.hz = fmaxf(bx.hz, sz[q]);
        }
        const float r2_prune = r2 * 1.00001f;
        for (int j = 0; j < cL; j += 2) {  // two independent loads in flight (the last may repeat a point)
            const float4 p0 = L[j], p1 = L[min(j + 1, cL - 1)];
            if (fminf(box_point_d2(bx, p0.x, p0.y, p0.z), box_point_d2(bx, p1.x, p1.y, p1.z)) > r2_prune) continue;
            bool h = false;
#pragma unroll
            for (int q = 0; q < BLK; q++) h |= (sqdist3(sx[q], sy[q], sz[q], p0.x, p0.y, p0.z) < r2) | (sqdist3(sx[q], sy[q], sz[q], p1.x, p1.y, p1.z) < r2);
            if (h) return true;
        }
    }
    return false;
}

__device__ __forceinline__ void phase_test(const FramePtrs& a, int cta, int G) {
    constexpr int kHardCap = MOR_HARD_CAP;
    __shared__ int s_edges, s_nhard, s_hard_hit[kHardCap];
    __shared__ int4 s_hard[kHardCap];
    __shared__ HeavyBoxes s_hard_box[kHardCap];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x == 0) { s_edges = 0; s_nhard = 0; }
    __syncthreads();
    const float r2 = a.r2;
    const int TL = min(__ldcg(&a.scratch->n_light), a.light_cap), TH = min(__ldcg(&a.scratch->n_heavy), a.heavy_cap);
    int2* eseg = a.edges + (size_t)cta * a.edge_seg;
    MOR_TRACE(16);
    // ---- light pairs: one thread each, 32 consecutive records per warp and step
    auto light_chunk = [&](int w0, int wend) {
        const int w = w0 + lane;
        bool hit = false;
        int sA = 0, sB = 0;
        if (w < wend) {
            const int2 lp = __ldcg(a.light + w);
            sA = lp.x & 0x1FFFFFF; sB = lp.y & 0x1FFFFFF;
            const int cA = (int)((unsigned)lp.x >> 25) + 1, cB = (int)((unsigned)lp.y >> 25) + 1;
            MOR_CHECK(sA + cA <= a.counts[MOR_CNT_NC] && sB + cB <= a.counts[MOR_CNT_NC], "light pair", sB);
            // the smaller cell (at most 16 points: the product is bounded) is held in registers, 4 or 8 points at a time,
            // and the larger one streams past it: one load per point of the larger cell and block instead of one per
            // test (the loads of 32 lanes go to 32 different lines: the L1 tag stage was the limit); the distance is
            // symmetric bit for bit, so the roles do not matter
            const bool a_small = cA <= cB;
            const float4* S = a.spts + (a_small ? sA : sB);
            const float4* L = a.spts + (a_small ? sB : sA);
            const int cS = a_small ? cA : cB, cL = a_small ? cB : cA;
            // all lines of the larger cell are requested now: the loop then finds them in L1 instead of paying an L2 round
            // trip every eight points
            for (int off = 128; off < cL * 16; off += 128) asm volatile("prefetch.global.L1 [%0];" ::"l"(reinterpret_cast<const char*>(L) + off));
            if (cS <= 4) hit = light_pair_connected<4>(S, cS, L, cL, r2);
            else hit = light_pair_connected<8>(S, cS, L, cL, r2);
        }
        if (hit) atomicMin(&a.hook[max(sA, sB)], min(sA, sB));
        const unsigned m = __ballot_sync(kFull, hit);
        if (m) {
            int slot = 0;
            if (lane == 0) slot = atomicAdd(&s_edges, __popc(m));
            slot = __shfl_sync(kFull, slot, 0) + __popc(m & ((1u << lane) - 1u));
            if (hit) { if (slot < a.edge_seg) eseg[slot] = make_int2(sA, sB); else atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_EDGE_CAP); }
        }
    };
    // ---- heavy pairs: one warp each, two pairs of a warp in flight together (their loads are the cost). The few pairs
    // that need the full scan are put aside and then taken on by the whole CTA, one chunk of B per warp: a single warp
    // would keep the group waiting for tens of microseconds on a pair of crowded cells.
    auto heavy_pairs = [&](int w, int w2, bool two) {
        int4 hp[2];
        hp[0] = __ldcg(a.heavy + w);
        hp[1] = two ? __ldcg(a.heavy + w2) : hp[0];
        float4 qa[2], qb[2];
#pragma unroll
        for (int q = 0; q < 2; q++) {
            MOR_CHECK(hp[q].x + hp[q].y <= a.counts[MOR_CNT_NC] && hp[q].z + hp[q].w <= a.counts[MOR_CNT_NC], "heavy pair", hp[q].z);
            qa[q] = a.spts[hp[q].x + (int)(((long long)lane * hp[q].y) >> 5)];
            qb[q] = a.spts[hp[q].z + (int)(((long long)lane * hp[q].w) >> 5)];
        }
#pragma unroll
        for (int q = 0; q < 2; q++) {
            if (q && !two) break;
            bool hit = heavy_probe(qa[q], qb[q], r2);
            if (!hit) {
                HeavyBoxes hb;
                if (heavy_boxes_apart(a, hp[q].x, hp[q].y, hp[q].z, hp[q].w, &hb, lane)) continue;
                int slot = kHardCap;
                if (lane == 0) slot = atomicAdd(&s_nhard, 1);
                slot = __shfl_sync(kFull, slot, 0);
                if (slot < kHardCap) { if (lane == 0) { s_hard[slot] = hp[q]; s_hard_box[slot] = hb; s_hard_hit[slot] = 0; } continue; }
                for (int b0 = 0; b0 < hp[q].w && !hit; b0 += 32) hit = heavy_scan_chunk(a, hb, hp[q].x, hp[q].y, hp[q].z, hp[q].w, b0, lane);  // (list full)
            }
            if (hit && lane == 0) {
                const int slot = atomicAdd(&s_edges, 1);
                if (slot < a.edge_seg) eseg[slot] = make_int2(hp[q].x, hp[q].z); else atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_EDGE_CAP);
                atomicMin(&a.hook[max(hp[q].x, hp[q].z)], min(hp[q].x, hp[q].z));
            }
        }
    };
    // Equal shares per CTA: the light pairs packed into the first warps (a warp issues the same instructions whether 12 or 32
    // of its lanes hold a pair: spreading them over all warps was 2x slower), the heavy pairs on the others, side by side.
    // (Dealing both lists out by ticket evens out the CTAs but queues every chunk on one word: 22.9 vs 16.1 us.)
    const int lper = (TL + G - 1) / G, llo = min(TL, cta * lper), lhi = min(TL, llo + lper);
    const int hper = (TH + G - 1) / G, hlo = min(TH, cta * hper), hhi = min(TH, hlo + hper);
    const int light_warps = min(kWarps, (lhi - llo + 31) >> 5);
    const int heavy_warps = max(kWarps - light_warps, 8);
    for (int base = llo + warp * 32; base < lhi; base += kT) light_chunk(base, lhi);
    MOR_TRACE_NOSYNC(17);
    const int hwarp = kWarps - 1 - warp;
    if (hwarp < heavy_warps)
        for (int w = hlo + hwarp; w < hhi; w += 2 * heavy_warps) heavy_pairs(w, w + heavy_warps, w + heavy_warps < hhi);
    __syncthreads();
    MOR_TRACE(18);
    const int nhard = min(s_nhard, kHardCap);
    if (nhard) {
        // work items (pair, chunk of B) in pair order, dealt out to the warps round-robin
        int item = warp;
        for (int p = 0, first = 0; p < nhard; p++) {
            const int4 hp = s_hard[p];
            const int chunks = (hp.w + 31) >> 5;
            if (item < first + chunks) {
                const HeavyBoxes hb = s_hard_box[p];
                for (; item < first + chunks; item += kWarps) {
                    // (another warp may already have found the pair connected: the flag only ever goes from 0 to 1; atomics keep the
                    // early exit free of a formal data race)
                    int seen = 0;
                    if (lane == 0) seen = atomicAdd(&s_hard_hit[p], 0);
                    if (__shfl_sync(kFull, seen, 0)) continue;
                    if (heavy_scan_chunk(a, hb, hp.x, hp.y, hp.z, hp.w, (item - first) * 32, lane) && lane == 0) atomicExch(&s_hard_hit[p], 1);
                }
            }
            first += chunks;
        }
        __syncthreads();
        for (int p = threadIdx.x; p < nhard; p += kT) {
            if (!s_hard_hit[p]) continue;
            const int4 hp = s_hard[p];
            const int slot = atomicAdd(&s_edges, 1);
            if (slot < a.edge_seg) eseg[slot] = make_int2(hp.x, hp.z); else atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_EDGE_CAP);
            atomicMin(&a.hook[max(hp.x, hp.z)], min(hp.x, hp.z));
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) a.edge_cnt[cta] = min(s_edges, a.edge_seg);
}

// ===================================================================================== phase E: components
// Connected components of the cell graph (a few thousand cells, ~8 edges per cell), then min <= size <= max
// (cpp:215-216) and the cluster order: size descending, min index ascending (A9 canonical rule).
// A union-find fed with all edges has every SM read and CAS the root words of the few big components: one L2 slice
// serves them one after the other, and that was most of the frame. Instead:
//  E1  the link phases left every cell pointing at its smallest connected neighbour: a spanning forest of local trees
//      (cells are numbered in scan order, so a surface is a handful of trees). Pointer jumping flattens it; the reads
//      are spread over the cells' own words.
//  E2  every edge compares the two labels (two scattered reads of non-shared words): all but a few hundred agree. The
//      rest are real unions between local trees (lock-free, roots ordered by index).
//  E3  every cell looks up its final root; size and minimum cloud index per root, grouped per warp before the atomics.
//  E4  one CTA selects and sorts the clusters (bitonic sort of (~size, min index) keys in shared memory).
__device__ __forceinline__ void phase_jump(const FramePtrs& a, int cta, int G) {
    int lo, hi;
    cta_slice(frame_vars().n_cells, cta, G, &lo, &hi);
    for (int i = lo + threadIdx.x; i < hi; i += kT) {
        const int node = a.cstart[i];
        int p = ld_parent(a.hook + node);
        MOR_CHECK(p >= 0 && p <= node, "jump p", p);
        while (true) {  // every cell jumps at the same time, so the distance to the root halves per step
            const int g = ld_parent(a.hook + p);
            if (g == p) break;
            st_parent(a.hook + node, g);
            p = g;
        }
    }
}

__device__ __forceinline__ void phase_cross(const FramePtrs& a, int cta, int G) {
    const int n = __ldcg(&a.edge_cnt[cta]);
    const int2* seg = a.edges + (size_t)cta * a.edge_seg;
    for (int e = threadIdx.x; e < n; e += kT) {
        const int2 uv = __ldcg(seg + e);
        MOR_CHECK(uv.x >= 0 && uv.x < a.counts[MOR_CNT_NC] && uv.y >= 0 && uv.y < a.counts[MOR_CNT_NC], "cross uv", uv.y);
        const int lu = ld_parent(a.hook + uv.x), lv = ld_parent(a.hook + uv.y);
        MOR_CHECK(lu >= 0 && lu < a.counts[MOR_CNT_NC] && lv >= 0 && lv < a.counts[MOR_CNT_NC], "cross label", lu);
        if (lu != lv) uf_union_pair(a.hook, lu, lv);
    }
}

__device__ __forceinline__ void phase_roots(const FramePtrs& a, int cta, int G) {
    int lo, hi;
    cta_slice(frame_vars().n_cells, cta, G, &lo, &hi);
    const int lane = threadIdx.x & 31;
    for (int base = lo; base < hi; base += kT) {
        const int i = base + threadIdx.x;
        const bool act = i < hi;
        int r = -1 - lane, cnt = 0, mn = 0x7FFFFFFF;
        if (act) {
            const int s0 = a.cstart[i];
            mn = __ldcg(&a.rmin[s0]);  // (the cell's own minimum, or already a smaller one of its component)
            cnt = a.ccnt[i];
            r = uf_find_ro(a.hook, s0);  // (no path halving here: nothing but the roots themselves may be stored in this phase)
            st_parent(a.hook + s0, r);   // flat for the per-point look-ups of the statistics phase
            if (r == s0) a.root_list[atomicAdd(&a.scratch->n_roots, 1)] = s0;
        }
        const unsigned grp = __match_any_sync(kFull, r);
        const int gsum = __reduce_add_sync(grp, cnt), gmin = __reduce_min_sync(grp, mn);
        if (act && (int)(__ffs(grp) - 1) == lane) { atomicAdd(&a.rsize[r], gsum); atomicMin(&a.rmin[r], gmin); }
    }
}

// Ascending sort of Pk (a power of two) keys in shared memory by the whole CTA.
__device__ __forceinline__ void bitonic_sort_smem(unsigned long long* keys, int Pk) {
    for (int size = 2; size <= Pk; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int t = threadIdx.x; t < (Pk >> 1); t += kT) {
                const int lo = 2 * t - (t & (stride - 1));
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const unsigned long long A = keys[lo], B = keys[hi];
                if ((A > B) == up) { keys[lo] = B; keys[hi] = A; }
            }
            __syncthreads();
        }
    }
}

__device__ __forceinline__ void phase_select(const FramePtrs& a, unsigned long long* keys) {
    __shared__ int s_k;
    const int n_roots = __ldcg(&a.scratch->n_roots);
    if (threadIdx.x == 0) s_k = 0;
    __syncthreads();
    for (int t = threadIdx.x; t < n_roots; t += kT) {
        const int i = a.root_list[t];
        const int sz = __ldcg(&a.rsize[i]), lab = __ldcg(&a.rmin[i]);
        if ((long long)sz >= a.min_cluster && (long long)sz <= a.max_cluster) {
            const int slot = atomicAdd(&s_k, 1);
            if (slot < a.kmax) keys[slot] = ((unsigned long long)(0xFFFFFFFFu - (unsigned)sz) << 32) | (unsigned)lab;
            else a.cid_of_root[lab] = -1;
        } else {
            a.cid_of_root[lab] = -1;
        }
    }
    __syncthreads();
    int K = s_k;
    if (K > a.kmax) {  // capacity exceeded: keep the first kmax found, flag the frame
        if (threadIdx.x == 0) atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_CLUSTER_CAP);
        K = a.kmax;
    }
    int Pk = 1;
    while (Pk < K) Pk <<= 1;
    for (int t = K + threadIdx.x; t < Pk; t += kT) keys[t] = ~0ull;
    __syncthreads();
    bitonic_sort_smem(keys, Pk);
    int nk = 0;
    for (int k = threadIdx.x; k < K; k += kT) {
        const unsigned long long kk = keys[k];
        const int root = (int)(unsigned)(kk & 0xFFFFFFFFull);
        const int sz = (int)(0xFFFFFFFFu - (unsigned)(kk >> 32));
        a.cl_root[k] = root; a.cl_size[k] = sz; a.cid_of_root[root] = k; a.cl_flags[k] = 0;
        nk += sz;
#pragma unroll
        for (int q = 0; q < 6; q++) a.acc_sum[k * 6 + q] = 0ull;
#pragma unroll
        for (int q = 0; q < 3; q++) { a.acc_box[k * 6 + q] = 0xFFFFFFFFu; a.acc_box[k * 6 + 3 + q] = 0u; }
    }
    atomicAdd(&a.counts[MOR_CNT_NK], nk);
    __syncthreads();
    // the same map by root position: the statistics phase then needs one dependent look-up less per point
    for (int t = threadIdx.x; t < n_roots; t += kT) {
        const int i = a.root_list[t];
        a.cid_of_pos[i] = __ldcg(&a.cid_of_root[__ldcg(&a.rmin[i])]);
    }
    if (threadIdx.x == 0) {
        a.counts[MOR_CNT_K] = K;
        const int e = __ldcg(&a.scratch->err_early);
        if (e) atomicOr(&a.counts[MOR_CNT_ERRFLAGS], e);
    }
}

// ---- large-K path of the select (out of line, like the other large-K steps: the frame kernels run at their register
// limit, and these rare steps should not add to it). Taken when the handle's kmax and the frame's root count (an upper bound on the
// size-valid clusters; final after the roots barrier, so every CTA of the group reads the same value) both exceed kSmallK.
template <bool LK>
__device__ __forceinline__ bool select_large(const FramePtrs& a) {
    return LK && __ldcg(&a.scratch->n_roots) > kSmallK;
}
// The same selection and order as phase_select, by the whole group: the size-valid keys go to a global array (capacity
// exceeded: the first kmax found are kept and the frame is flagged, as in phase_select), runs of up to kSmallK keys are
// sorted in shared memory (bitonic), then merged in pairs between group barriers - every key finds its place by a binary
// search in the other run (the keys are unique: the labels are). Every CTA must call; writes what phase_select writes.
__device__ __noinline__ void phase_select_large(const FramePtrs& a, int cta, int G, unsigned long long* dyn, GroupBarrier& bar) {
    const int n_roots = __ldcg(&a.scratch->n_roots);
    const int gtid = cta * kT + threadIdx.x, stride = G * kT;
    unsigned long long* src = a.sort_keys;
    unsigned long long* dst = a.sort_keys + a.kmax;
    for (int t = gtid; t < n_roots; t += stride) {
        const int i = __ldcg(&a.root_list[t]);
        const int sz = __ldcg(&a.rsize[i]), lab = __ldcg(&a.rmin[i]);
        if ((long long)sz >= a.min_cluster && (long long)sz <= a.max_cluster) {
            const int slot = atomicAdd(&a.scratch->n_sel, 1);
            if (slot < a.kmax) src[slot] = ((unsigned long long)(0xFFFFFFFFu - (unsigned)sz) << 32) | (unsigned)lab;
            else a.cid_of_root[lab] = -1;
        } else {
            a.cid_of_root[lab] = -1;
        }
    }
    bar.sync();
    const int found = __ldcg(&a.scratch->n_sel);
    const int K = min(found, a.kmax);
    int R = kSmallK;  // run length: what the dynamic shared memory holds
    while ((size_t)R * sizeof(unsigned long long) > (size_t)a.frame_smem) R >>= 1;
    for (int r = cta; (long long)r * R < K; r += G) {
        const int b0 = r * R, len = min(R, K - b0);
        int Pk = 1;
        while (Pk < len) Pk <<= 1;
        for (int t = threadIdx.x; t < Pk; t += kT) dyn[t] = t < len ? __ldcg(&src[b0 + t]) : ~0ull;
        __syncthreads();
        bitonic_sort_smem(dyn, Pk);
        for (int t = threadIdx.x; t < len; t += kT) src[b0 + t] = dyn[t];
        __syncthreads();
    }
    for (int w = R; w < K; w <<= 1) {
        bar.sync();
        for (int e = gtid; e < K; e += stride) {
            const unsigned long long x = __ldcg(&src[e]);
            const int b = e / (2 * w) * (2 * w);
            const bool in_a = e < b + w;
            const int o0 = in_a ? min(b + w, K) : b, o1 = in_a ? min(b + 2 * w, K) : b + w;  // the other run
            int lo = o0, hi = o1;
            while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldcg(&src[mid]) < x) lo = mid + 1; else hi = mid;
            }
            dst[b + (e - (in_a ? b : b + w)) + (lo - o0)] = x;
        }
        unsigned long long* t = src; src = dst; dst = t;
    }
    bar.sync();
    int nk = 0;
    for (int k = gtid; k < K; k += stride) {
        const unsigned long long kk = __ldcg(&src[k]);
        const int root = (int)(unsigned)(kk & 0xFFFFFFFFull);
        const int sz = (int)(0xFFFFFFFFu - (unsigned)(kk >> 32));
        a.cl_root[k] = root; a.cl_size[k] = sz; a.cid_of_root[root] = k; a.cl_flags[k] = 0;
        nk += sz;
#pragma unroll
        for (int q = 0; q < 6; q++) a.acc_sum[k * 6 + q] = 0ull;
#pragma unroll
        for (int q = 0; q < 3; q++) { a.acc_box[k * 6 + q] = 0xFFFFFFFFu; a.acc_box[k * 6 + 3 + q] = 0u; }
    }
    nk = __reduce_add_sync(kFull, nk);
    if ((threadIdx.x & 31) == 0 && nk) atomicAdd(&a.counts[MOR_CNT_NK], nk);
    bar.sync();
    for (int t = gtid; t < n_roots; t += stride) {
        const int i = __ldcg(&a.root_list[t]);
        a.cid_of_pos[i] = __ldcg(&a.cid_of_root[__ldcg(&a.rmin[i])]);
    }
    if (gtid == 0) {
        a.counts[MOR_CNT_K] = K;
        int e = __ldcg(&a.scratch->err_early);
        if (found > a.kmax) e |= ERR_CLUSTER_CAP;
        if (e) atomicOr(&a.counts[MOR_CNT_ERRFLAGS], e);
    }
}

// ===================================================================================== phase G: cluster statistics
// Per-cluster statistics (cpp:221-244): cluster id of every point, exact coordinate sums for
// compute3DCentroid<double> (A10) and getMinMax3D bounding boxes (cpp:272-275). Needs the selection (cid_of_pos) and
// nothing of the match: a pipelined launch runs it at the start of the back half, so the front half ends at the select.
// One point's statistics in the same kind of steps: the point and its cell's node, the node's root (hook is flat), the
// root's label and cluster id, then the stores.
struct StatsItem { float4 p; int x, lab, k; };
__device__ __forceinline__ void stats_load(const FramePtrs& a, int s, int hi, StatsItem& it) {
    it.p = make_float4(0, 0, 0, 0); it.k = -1;
    if (s < hi) { it.p = a.spts[s]; it.x = a.slead[s]; }
}
__device__ __forceinline__ void stats_root(const FramePtrs& a, int s, int hi, StatsItem& it) {
    if (s < hi) it.x = a.hook[it.x];  // consecutive points share these words
}
__device__ __forceinline__ void stats_lookup(const FramePtrs& a, int s, int hi, StatsItem& it) {
    if (s < hi) { it.lab = a.rmin[it.x]; it.k = a.cid_of_pos[it.x]; }
}
__device__ __forceinline__ void stats_finish(const FramePtrs& a, int s, int hi, int nc, const StatsItem& it) {
    if (s >= hi) return;
    const int c = __float_as_int(it.p.w);
    MOR_CHECK(it.lab >= 0 && it.lab < nc, "label", it.lab);
    a.label[c] = it.lab;
    a.cid[c] = it.k;
    a.scid[s] = it.k;
}
__device__ __forceinline__ void phase_stats(const FramePtrs& a, int cta, int G) {
    const int nc = frame_vars().nc;
    int lo, hi;
    cta_slice(nc, cta, G, &lo, &hi);
    for (int base = lo; base < hi; base += kT) {
        const int s = base + threadIdx.x;
        StatsItem it;
        stats_load(a, s, hi, it);
        stats_root(a, s, hi, it);
        stats_lookup(a, s, hi, it);
        stats_finish(a, s, hi, nc, it);
        block_cluster_accumulate<true>(a.acc_sum, a.acc_box, it.k, it.k >= 0, it.p.x, it.p.y, it.p.z);
    }
}
// The pipelined back half's first phase: the previous clusters' transform (transform_range) and this frame's
// statistics (phase_stats) in one loop, step by step, so that a round waits for the two chains of dependent loads side
// by side instead of one after the other.
template <bool LK>
__device__ __forceinline__ void stats_transform(const FramePtrs& a, int cta, int G) {
    const int nc = frame_vars().nc;
    const bool wide = lattice_wide<LK>(a);
    int lo_s, hi_s, lo_t = 0, hi_t = 0;
    cta_slice(nc, cta, G, &lo_s, &hi_s);
    if (a.two_frames) cta_slice(a.p_counts[MOR_CNT_NC], cta, G, &lo_t, &hi_t);
    for (int r = 0; lo_s + r < hi_s || lo_t + r < hi_t; r += kT) {  // (uniform over the CTA)
        const int s = lo_s + r + threadIdx.x, t = lo_t + r + threadIdx.x;
        StatsItem is;
        XformItem ix;
        stats_load(a, s, hi_s, is);
        xform_load(a, t, hi_t, ix);
        stats_root(a, s, hi_s, is);
        xform_lookup(a, t, hi_t, ix);
        stats_lookup(a, s, hi_s, is);
        xform_finish(a, t, hi_t, wide, ix);
        stats_finish(a, s, hi_s, nc, is);
        block_cluster_accumulate<false>(nullptr, a.pacc_box, ix.k, ix.k >= 0, ix.t.x, ix.t.y, ix.t.z);
        block_cluster_accumulate<true>(a.acc_sum, a.acc_box, is.k, is.k >= 0, is.p.x, is.p.y, is.p.z);
    }
}


// Block-wide ordered compaction helper for the single-CTA phases: returns the exclusive rank of `flag` among all
// threads, *total = number of set flags. kSingle threads.
__device__ __forceinline__ int single_block_rank(bool flag, int* total) {
    __shared__ int s_w[kSingle / 32];
    __shared__ int s_tot;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const unsigned m = __ballot_sync(kFull, flag);
    if (lane == 0) s_w[warp] = __popc(m);
    __syncthreads();
    if (warp == 0) {
        int v = s_w[lane], inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int t = __shfl_up_sync(kFull, inc, o);
            if (lane >= o) inc += t;
        }
        s_w[lane] = inc - v;
        if (lane == 31) s_tot = inc;
    }
    __syncthreads();
    const int r = s_w[warp] + __popc(m & ((1u << lane) - 1u));
    *total = s_tot;
    __syncthreads();
    return r;
}

// ===================================================================================== phase H: match (one CTA)
// Finalise centroids/boxes, transform the previous centroids (cpp:540-541), reciprocal 1-NN between centroid sets
// (cpp:291-294, A16), volume constraint (cpp:264-283, A17).
__device__ __forceinline__ int nn_brute(const float* pts, int n, float qx, float qy, float qz, float* out_d) {
    int best = -1;
    float bd = 3.402823466e+38f;
    for (int i = 0; i < n; i++) {
        const float d = sqdist3(qx, qy, qz, pts[i * 3], pts[i * 3 + 1], pts[i * 3 + 2]);
        if (d < bd) { bd = d; best = i; }  // ties -> lowest index
    }
    *out_d = bd;
    return best;
}

// The working set (centroids, boxes, the reciprocal list) lives in shared memory when the frame has few enough clusters
// for it (a few hundred: every LiDAR frame) - the step is a chain of small dependent passes, and each pass through
// global memory would cost a round trip; every result is written to its global array as well.
constexpr int kMatchBytesPerCluster = (3 + 6 + 3 + 6 + 3) * 4;
// The same search by a whole warp (lanes across the candidates): equal distances go to the lowest index, like the
// sequential scan; -1 if no candidate compares below FLT_MAX. The result is valid in every lane.
__device__ __forceinline__ int nn_warp(const float* pts, int n, float qx, float qy, float qz, float* out_d, int lane) {
    int best = -1;
    float bd = 3.402823466e+38f;
    for (int i = lane; i < n; i += 32) {
        const float d = sqdist3(qx, qy, qz, pts[i * 3], pts[i * 3 + 1], pts[i * 3 + 2]);
        if (d < bd) { bd = d; best = i; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const float od = __shfl_xor_sync(kFull, bd, o);
        const int ob = __shfl_xor_sync(kFull, best, o);
        if (ob >= 0 && (best < 0 || od < bd || (od == bd && ob < best))) { bd = od; best = ob; }
    }
    *out_d = bd;
    return best;
}

template <bool FAST, bool FINALIZE = true>
__device__ __forceinline__ void phase_match_impl(const FramePtrs& a, unsigned long long* dyn) {
    const int K = a.counts[MOR_CNT_K];
    const int Kp = a.two_frames ? a.p_counts[MOR_CNT_K] : 0;
    constexpr int kNnBytes = kSingle * 12;  // (ok, match, distance) of one chunk of queries
    const int cap = (a.frame_smem - kNnBytes) / kMatchBytesPerCluster;
    constexpr bool fast = FAST;
    const int cta = 0; (void)cta;
    MOR_TRACE(19);
    float* const sm = reinterpret_cast<float*>(dyn);
    // (no run-time choice between the two homes of an array: the compiler must see which address space a load goes to)
    float *cc, *cb, *pc, *pb, *rd;
    int *rq, *rm;
    if (FAST) {
        cc = sm; cb = sm + 3 * cap; pc = sm + 9 * cap; pb = sm + 12 * cap;       // [K][3], [K][6], [Kp][3], [Kp][6]
        rq = reinterpret_cast<int*>(sm + 18 * cap); rm = reinterpret_cast<int*>(sm + 19 * cap); rd = sm + 20 * cap;
    } else {
        cc = a.cl_centroid; cb = a.cl_bbox; pc = a.pct; pb = a.pbbox; rq = a.recip_q; rm = a.recip_m; rd = a.match_dist;
    }
    int* const nn_j = reinterpret_cast<int*>(sm + 21 * cap);  // [kSingle] each: the chunk's nearest neighbour, its distance, reciprocal?
    float* const nn_d = sm + 21 * cap + kSingle;
    int* const nn_ok = reinterpret_cast<int*>(sm + 21 * cap + 2 * kSingle);
    // the current clusters are finalised by the first half of the CTA while the second half brings the previous ones over
    // (two chains of dependent loads side by side)
    const int half = kSingle / 2;
    for (int c = threadIdx.x; c < K && threadIdx.x < half; c += half) {
        const double n = (double)a.cl_size[c];
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const float v = FINALIZE ? (float)join_fixed_mean((long long)__ldcg(&a.acc_sum[c * 6 + q * 2]), (long long)__ldcg(&a.acc_sum[c * 6 + q * 2 + 1]), n)
                                     : __ldcg(&a.cl_centroid[c * 3 + q]);
            if (FINALIZE) a.cl_centroid[c * 3 + q] = v;
            if (fast) cc[c * 3 + q] = v;
        }
#pragma unroll
        for (int q = 0; q < 6; q++) {
            const float v = FINALIZE ? fkey_inv(__ldcg(&a.acc_box[c * 6 + q])) : __ldcg(&a.cl_bbox[c * 6 + q]);
            if (FINALIZE) a.cl_bbox[c * 6 + q] = v;
            if (fast) cb[c * 6 + q] = v;
        }
    }
    if (!a.two_frames) return;
    // previous centroids and boxes into the current frame
    for (int i = (int)threadIdx.x - half; i >= 0 && i < Kp; i += half) {
        const float3 t = xform(a.M, a.p_cl_centroid[i * 3], a.p_cl_centroid[i * 3 + 1], a.p_cl_centroid[i * 3 + 2]);
        a.pct[i * 3] = t.x; a.pct[i * 3 + 1] = t.y; a.pct[i * 3 + 2] = t.z;
        if (fast) { pc[i * 3] = t.x; pc[i * 3 + 1] = t.y; pc[i * 3 + 2] = t.z; }
#pragma unroll
        for (int q = 0; q < 6; q++) {
            const float v = fkey_inv(__ldcg(&a.pacc_box[i * 6 + q]));
            a.pbbox[i * 6 + q] = v;
            if (fast) pb[i * 6 + q] = v;
        }
        a.match_of_prev[i] = -1; a.mid_of_prev[i] = -1;
    }
    for (int j = threadIdx.x; j < K; j += kSingle) a.mid_of_cur[j] = -1;
    __syncthreads();
    MOR_TRACE(20);
    // reciprocal correspondences, ascending query index
    int n_recip = 0;
    for (int base = 0; base < Kp; base += kSingle) {
        {   // a warp per query: nearest current cluster, then that cluster's nearest previous one
            const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
            for (int u = warp; u < kSingle && base + u < Kp; u += kWarps) {
                const int q = base + u;
                float dq = 0.f, dr;
                int jq = -1, ir = -1;
                if (K > 0) {
                    jq = nn_warp(cc, K, pc[q * 3], pc[q * 3 + 1], pc[q * 3 + 2], &dq, lane);
                    ir = nn_warp(pc, Kp, cc[jq * 3], cc[jq * 3 + 1], cc[jq * 3 + 2], &dr, lane);
                }
                if (lane == 0) { nn_j[u] = jq; nn_d[u] = dq; nn_ok[u] = (K > 0 && ir == q) ? 1 : 0; }
            }
        }
        MOR_TRACE(23);
        __syncthreads();
        const int i = base + threadIdx.x;
        bool ok = false; int j = -1; float d = 0.f;
        if (i < Kp) { ok = nn_ok[threadIdx.x] != 0; j = nn_j[threadIdx.x]; d = nn_d[threadIdx.x]; }
        int tot;
        const int r = single_block_rank(ok, &tot);
        if (ok) {
            rq[n_recip + r] = i; rm[n_recip + r] = j; rd[n_recip + r] = d;
            if (fast) { a.recip_q[n_recip + r] = i; a.recip_m[n_recip + r] = j; }
        }
        n_recip += tot;
    }
    __syncthreads();
    MOR_TRACE(21);
    // volume constraint (slow path: match_dist is rewritten in place - rank <= index, chunked with barriers)
    int n_match = 0;
    for (int base = 0; base < n_recip; base += kSingle) {
        const int u = base + threadIdx.x;
        bool ok = false; int i = -1, j = -1; float d = 0.f;
        if (u < n_recip) {
            i = rq[u]; j = rm[u]; d = rd[u];
            const float* bp = pb + i * 6; const float* bc = cb + j * 6;
            const double volp = (double)__fmul_rn(__fmul_rn(__fsub_rn(bp[3], bp[0]), __fsub_rn(bp[4], bp[1])), __fsub_rn(bp[5], bp[2]));
            const double volc = (double)__fmul_rn(__fmul_rn(__fsub_rn(bc[3], bc[0]), __fsub_rn(bc[4], bc[1])), __fsub_rn(bc[5], bc[2]));
            ok = (fabs(volp - volc) / (volp + volc)) < (double)a.volume_constraint;  // NaN -> false
        }
        int tot;
        const int r = single_block_rank(ok, &tot);
        if (ok) {
            const int m = n_match + r;
            a.match_q[m] = i; a.match_m[m] = j; a.match_dist[m] = d;
            a.match_of_prev[i] = j; a.mid_of_prev[i] = m; a.mid_of_cur[j] = m;
            a.newcount[m] = 0; a.match_score[m] = 0.0;
            atomicAdd(&a.counts[MOR_CNT_P1], a.p_cl_size[i]);
            atomicAdd(&a.counts[MOR_CNT_P2], a.cl_size[j]);
        }
        n_match += tot;
    }
    MOR_TRACE(22);
    if (threadIdx.x == 0) {
        a.counts[MOR_CNT_MU] = n_recip; a.counts[MOR_CNT_M] = n_match;
        a.counts[MOR_CNT_NKPREV] = a.p_counts[MOR_CNT_NK];
    }
}

__device__ __forceinline__ void phase_match(const FramePtrs& a, unsigned long long* dyn) {
    const int K = a.counts[MOR_CNT_K];
    const int Kp = a.two_frames ? a.p_counts[MOR_CNT_K] : 0;
    const int cap = (a.frame_smem - kSingle * 12) / kMatchBytesPerCluster;
    if (K <= cap && Kp <= cap) phase_match_impl<true>(a, dyn); else phase_match_impl<false>(a, dyn);
}

// ---- large-K path of the match: taken when either frame has more than kSmallK clusters (both counts are final before
// the match, so the choice is the same in every CTA of the group).
template <bool LK>
__device__ __forceinline__ bool match_large(const FramePtrs& a) {
    return LK && (__ldcg(&a.counts[MOR_CNT_K]) > kSmallK || (a.two_frames && __ldcg(&a.p_counts[MOR_CNT_K]) > kSmallK));
}
// Nearest neighbour of up to kNnQ queries (q0 ... q0 + nq - 1 of qpts, [.][3]) among the n points cand ([n][3]), by one
// CTA: the candidates pass through shared memory in tiles of kNnTile, and each quarter of the CTA scans its own quarter of
// every tile for all queries. Equal distances go to the lowest index, like nn_warp and the reference's linear scan (a
// quarter scans its indices in ascending order, the quarters are merged by index); -1 / FLT_MAX if no candidate compares
// below FLT_MAX. Results to out_k[q0 + u] (and out_d). tile: kNnTile float4 of shared memory. Every thread must call.
constexpr int kNnQ = 256, kNnParts = kT / kNnQ, kNnTile = 4096;
__device__ __forceinline__ void nn_chunk(const float* qpts, int q0, int nq, const float* cand, int n, float4* tile, int* out_k, float* out_d) {
    const int u = threadIdx.x % kNnQ, part = threadIdx.x / kNnQ;
    float qx = 0.f, qy = 0.f, qz = 0.f;
    if (u < nq) { qx = __ldcg(qpts + (size_t)(q0 + u) * 3); qy = __ldcg(qpts + (size_t)(q0 + u) * 3 + 1); qz = __ldcg(qpts + (size_t)(q0 + u) * 3 + 2); }
    int best = -1;
    float bd = 3.402823466e+38f;
    for (int t0 = 0; t0 < n; t0 += kNnTile) {
        const int m = min(kNnTile, n - t0);
        __syncthreads();  // the previous tile's readers are done
        for (int t = threadIdx.x; t < m; t += kT) {
            const float* c = cand + (size_t)(t0 + t) * 3;
            tile[t] = make_float4(__ldcg(c), __ldcg(c + 1), __ldcg(c + 2), 0.f);
        }
        __syncthreads();
        const int hi = min(m, (part + 1) * (kNnTile / kNnParts));
        for (int i = part * (kNnTile / kNnParts); i < hi; i++) {
            const float4 c = tile[i];
            const float d = sqdist3(qx, qy, qz, c.x, c.y, c.z);
            if (d < bd) { bd = d; best = t0 + i; }
        }
    }
    __syncthreads();
    int* const sk = reinterpret_cast<int*>(tile);
    float* const sd = reinterpret_cast<float*>(tile) + kT;
    sk[threadIdx.x] = best; sd[threadIdx.x] = bd;
    __syncthreads();
    if (part == 0 && u < nq) {
        for (int p = 1; p < kNnParts; p++) {
            const int ob = sk[p * kNnQ + u];
            const float od = sd[p * kNnQ + u];
            if (ob >= 0 && (best < 0 || od < bd || (od == bd && ob < best))) { bd = od; best = ob; }
        }
        out_k[q0 + u] = best;
        if (out_d) out_d[q0 + u] = bd;
    }
    __syncthreads();
}

// phase_match_impl by the whole group: finalise centroids and boxes and transform the previous ones (spread over the
// group), barrier, nearest current cluster of every previous one and nearest previous cluster of every current one
// (chunks of queries dealt out over the CTAs), barrier, then one CTA keeps the reciprocal pairs in ascending query index
// and applies the volume constraint in that order: the arrays and counts phase_match_impl writes. Every CTA must call;
// the caller's barrier follows.
__device__ __noinline__ void phase_match_large(const FramePtrs& a, int cta, int G, unsigned long long* dyn, GroupBarrier& bar) {
    const int K = __ldcg(&a.counts[MOR_CNT_K]);
    const int Kp = a.two_frames ? __ldcg(&a.p_counts[MOR_CNT_K]) : 0;
    const int gtid = cta * kT + threadIdx.x, stride = G * kT;
    for (int c = gtid; c < K; c += stride) {
        const double n = (double)__ldcg(&a.cl_size[c]);
#pragma unroll
        for (int q = 0; q < 3; q++)
            a.cl_centroid[c * 3 + q] = (float)join_fixed_mean((long long)__ldcg(&a.acc_sum[c * 6 + q * 2]), (long long)__ldcg(&a.acc_sum[c * 6 + q * 2 + 1]), n);
#pragma unroll
        for (int q = 0; q < 6; q++) a.cl_bbox[c * 6 + q] = fkey_inv(__ldcg(&a.acc_box[c * 6 + q]));
    }
    if (!a.two_frames) return;
    for (int i = gtid; i < Kp; i += stride) {
        const float3 t = xform(a.M, a.p_cl_centroid[i * 3], a.p_cl_centroid[i * 3 + 1], a.p_cl_centroid[i * 3 + 2]);
        a.pct[i * 3] = t.x; a.pct[i * 3 + 1] = t.y; a.pct[i * 3 + 2] = t.z;
#pragma unroll
        for (int q = 0; q < 6; q++) a.pbbox[i * 6 + q] = fkey_inv(__ldcg(&a.pacc_box[i * 6 + q]));
        a.match_of_prev[i] = -1; a.mid_of_prev[i] = -1;
    }
    for (int j = gtid; j < K; j += stride) a.mid_of_cur[j] = -1;
    bar.sync();
    float4* const tile = reinterpret_cast<float4*>(dyn);
    const int chunks_prev = (Kp + kNnQ - 1) / kNnQ, chunks_cur = (K + kNnQ - 1) / kNnQ;
    for (int c = cta; c < chunks_prev + chunks_cur; c += G) {
        if (c < chunks_prev) nn_chunk(a.pct, c * kNnQ, min(kNnQ, Kp - c * kNnQ), a.cl_centroid, K, tile, a.nn_cur, a.nn_dist);
        else { const int q0 = (c - chunks_prev) * kNnQ; nn_chunk(a.cl_centroid, q0, min(kNnQ, K - q0), a.pct, Kp, tile, a.nn_prev, nullptr); }
    }
    bar.sync();
    if (cta != 0) return;
    int n_recip = 0, n_match = 0;
    for (int base = 0; base < Kp; base += kSingle) {
        const int i = base + threadIdx.x;
        bool ok = false, vok = false;
        int j = -1;
        float d = 0.f;
        if (i < Kp) {
            j = __ldcg(&a.nn_cur[i]); d = __ldcg(&a.nn_dist[i]);
            ok = j >= 0 && __ldcg(&a.nn_prev[j]) == i;
            if (ok) {
                const float* bp = a.pbbox + i * 6; const float* bc = a.cl_bbox + j * 6;
                const double volp = (double)__fmul_rn(__fmul_rn(__fsub_rn(__ldcg(bp + 3), __ldcg(bp)), __fsub_rn(__ldcg(bp + 4), __ldcg(bp + 1))), __fsub_rn(__ldcg(bp + 5), __ldcg(bp + 2)));
                const double volc = (double)__fmul_rn(__fmul_rn(__fsub_rn(__ldcg(bc + 3), __ldcg(bc)), __fsub_rn(__ldcg(bc + 4), __ldcg(bc + 1))), __fsub_rn(__ldcg(bc + 5), __ldcg(bc + 2)));
                vok = (fabs(volp - volc) / (volp + volc)) < (double)a.volume_constraint;  // NaN -> false
            }
        }
        int tot;
        const int r = single_block_rank(ok, &tot);
        if (ok) { a.recip_q[n_recip + r] = i; a.recip_m[n_recip + r] = j; }
        n_recip += tot;
        const int rm = single_block_rank(vok, &tot);
        if (vok) {
            const int m = n_match + rm;
            a.match_q[m] = i; a.match_m[m] = j; a.match_dist[m] = d;
            a.match_of_prev[i] = j; a.mid_of_prev[i] = m; a.mid_of_cur[j] = m;
            a.newcount[m] = 0; a.match_score[m] = 0.0;
            atomicAdd(&a.counts[MOR_CNT_P1], a.p_cl_size[i]);
            atomicAdd(&a.counts[MOR_CNT_P2], __ldcg(&a.cl_size[j]));
        }
        n_match += tot;
    }
    if (threadIdx.x == 0) {
        a.counts[MOR_CNT_MU] = n_recip; a.counts[MOR_CNT_M] = n_match;
        a.counts[MOR_CNT_NKPREV] = a.p_counts[MOR_CNT_NK];
    }
}
// ===================================================================================== phase I: moving test
// Method 2 (default): the score of a matched pair is the number of points of the current cluster whose octree leaf
// holds no point of the transformed previous cluster (cpp:325-330).
template <bool LK>
__device__ __forceinline__ void phase_lattice_count(const FramePtrs& a, int cta, int G) {
    int lo, hi;
    cta_slice(frame_vars().nc, cta, G, &lo, &hi);
    const int lane = threadIdx.x & 31;
    const bool wide = LK && a.p_counts[MOR_CNT_K] > kLatticeNarrowK;
    for (int base = lo; base < hi; base += kT) {
        const int s = base + threadIdx.x;
        int m = -1;
        bool is_new = false;
        if (s < hi) {
            const int k = a.scid[s];
            m = k >= 0 ? a.mid_of_cur[k] : -1;
            if (m >= 0) {
                const float4 p = a.spts[s];
                const int kp = a.match_q[m];
                unsigned long long key;
                if (lattice_key(a.anchorp + (size_t)kp * 3, kp, p.x, p.y, p.z, &key, wide)) is_new = !hset_contains(a.lattice, a.lattice_mask, key);
                else { atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_LATTICE_RANGE); is_new = true; }
            }
        }
        const unsigned same = __match_any_sync(kFull, is_new ? m : -1 - lane);
        if (is_new && (int)(__ffs(same) - 1) == lane) atomicAdd(&a.newcount[m], __popc(same));
    }
}

// Method 1: CorrespondenceEstimation::determineCorrespondences (cpp:343-361): for every point of the transformed
// previous cluster the nearest point of the matched current cluster; only squared distances inside (pde_lb, pde_ub)
// count, so the search is bounded by sqrt(pde_ub) on the clustering grid. Shells of growing Chebyshev distance around
// the query's cell: a point in shell r is at least (r-1)*h away, so the search stops as soon as that bound exceeds the
// best distance (or pde_ub: farther neighbours never count), and a neighbour at d2 <= pde_lb settles the answer.
__device__ __forceinline__ void phase_pde_count(const FramePtrs& a, int cta, int G) {
    const int ncp = a.p_counts[MOR_CNT_NC];
    const int ring = a.pde_ring;
    const float h = (float)a.cell_h;
    for (int base = cta * kT; base < ncp; base += G * kT) {
        const int c = base + threadIdx.x;
        if (c >= ncp) continue;
        const float4 t = a.tpts[c];
        const int kp = __float_as_int(t.w);
        const int m = kp >= 0 ? a.mid_of_prev[kp] : -1;
        if (m < 0) continue;
        const int target = a.match_m[m];
        bool oob = false;
        const int cx = cell_coord(t.x, a.inv_h, &oob), cy = cell_coord(t.y, a.inv_h, &oob), cz = cell_coord(t.z, a.inv_h, &oob);
        float best = 3.402823466e+38f;
        bool settled = oob;  // a query outside the grid's range has no neighbour within sqrt(pde_ub)
        for (int r = 0; r <= ring && !settled; r++) {
            if (r > 1) {
                const float lb = (float)(r - 1) * h * 0.99999f;
                if (lb * lb >= fminf(best, a.pde_ub)) break;
            }
            for (int dz = -r; dz <= r && !settled; dz++)
                for (int dy = -r; dy <= r && !settled; dy++) {
                    const bool face = (dz == -r || dz == r || dy == -r || dy == r);  // rows on the shell's faces: whole x-run
                    const int step = (face || r == 0) ? 1 : 2 * r;                    // otherwise only the two end cells
                    for (int dx = -r; dx <= r; dx += step) {
                        Cell e;
                        if (!grid_lookup(a, cell_pack(cx + dx, cy + dy, cz + dz), &e)) continue;
                        for (int j = e.start; j < e.start + e.cnt; j++) {
                            if (a.scid[j] != target) continue;
                            const float4 q = a.spts[j];
                            best = fminf(best, sqdist3(t.x, t.y, t.z, q.x, q.y, q.z));
                        }
                        if (best <= a.pde_lb) { settled = true; break; }
                    }
                }
        }
        if (best > a.pde_lb && best < a.pde_ub) atomicAdd(&a.newcount[m], 1);
    }
}

// ===================================================================================== phase J: chain (one CTA) + cleanup
// Detection flags (cpp:580-606) and the N-frame consistency chain: checkMovingClusterChain (cpp:478-514),
// recurseFindClusterChain (cpp:415-453), pushCentroid (cpp:455-476). corrs_vec / res_vec are device-resident ring
// buffers; a correspondence map is stored as match_of_prev[].
__device__ __forceinline__ void phase_chain(const FramePtrs& a) {
    const int K = a.counts[MOR_CNT_K], Kp = a.p_counts[MOR_CNT_K], M = a.counts[MOR_CNT_M];
    const int D = a.ring_depth, kmax = a.kmax;
    TrackState* ts = a.track;
    __shared__ int s_flag_any;
    const int cta = 0; (void)cta;
    MOR_TRACE(24);
    for (int m = threadIdx.x; m < M; m += kSingle) {
        const unsigned long long n1 = (unsigned long long)a.p_cl_size[a.match_q[m]], n2 = (unsigned long long)a.cl_size[a.match_m[m]];
        double score, thr;
        if (a.method == 1) {
            score = (double)__ldcg(&a.newcount[m]) / (double)((n1 + n2) / 2ull);  // cpp:361
            thr = (double)a.pde_thr;                                       // cpp:586
        } else {
            score = (double)__ldcg(&a.newcount[m]);                                        // cpp:330
            thr = (double)((n1 + n2) / (unsigned long long)(long long)a.opc_factor);      // cpp:590, unsigned division
        }
        a.match_score[m] = score;
        a.cl_flags[a.match_m[m]] = score > thr ? 1 : 0;
    }
    __syncthreads();
    // ---- checkMovingClusterChain: push buffers
    const int corr_slot = (ts->corr_head + ts->corr_count) % D;
    for (int i = threadIdx.x; i < Kp; i += kSingle) a.corr_ring[corr_slot * kmax + i] = a.match_of_prev[i];
    int res_count = ts->res_count;
    const int res_head = ts->res_head;
    if (res_count == 0) {
        const int slot = res_head % D;
        for (int i = threadIdx.x; i < Kp; i += kSingle) a.res_ring[slot * kmax + i] = a.p_cl_flags[i];
        if (threadIdx.x == 0) a.res_len[slot] = Kp;
        res_count = 1;
    }
    {
        const int slot = (res_head + res_count) % D;
        for (int j = threadIdx.x; j < K; j += kSingle) a.res_ring[slot * kmax + j] = a.cl_flags[j];
        if (threadIdx.x == 0) a.res_len[slot] = K;
        res_count += 1;
    }
    if (threadIdx.x == 0) a.corr_len[corr_slot] = Kp;
    const int corr_count = ts->corr_count + 1;
    const int corr_head = ts->corr_head;
    __syncthreads();
    MOR_TRACE(25);
    float* const mo_centroid = a.mo_centroid + (size_t)a.mo_parity * a.momax * 3;
    int* const mo_conf = a.mo_conf + (size_t)a.mo_parity * a.momax;
    int n_mo = ts->n_mo[a.mo_parity];
    if (res_count >= a.moving_confidence) {
        const int r0 = res_head % D;
        const int len0 = a.res_len[r0];
        // every flagged cluster of the oldest frame is followed through all buffered maps
        for (int i = threadIdx.x; i < len0; i += kSingle) {
            int track = -1;
            if (a.res_ring[r0 * kmax + i]) {
                track = i;
                for (int col = 0; col < corr_count && track >= 0; col++) {
                    const int cs = (corr_head + col) % D;
                    const int j = track < a.corr_len[cs] ? a.corr_ring[cs * kmax + track] : -1;
                    const int rs = (res_head + col + 1) % D;
                    track = (j >= 0 && a.res_ring[rs * kmax + j]) ? j : -1;
                }
            }
            a.found[i] = track;
        }
        __syncthreads();
        // keep the surviving chain ends, in ascending i (in place: write index <= read index)
        int n_found = 0;
        for (int base = 0; base < len0; base += kSingle) {
            const int i = base + threadIdx.x;
            const int f = i < len0 ? a.found[i] : -1;
            int tot;
            const int r = single_block_rank(f >= 0, &tot);
            if (f >= 0) a.found[n_found + r] = f;
            n_found += tot;
            __syncthreads();
        }
        MOR_TRACE(26);
        // pushCentroid in that order; the scan over mo_vec is parallel, the append is serial
        for (int i = 0; i < n_found; i++) {
            const int f = a.found[i];
            const float px = a.cl_centroid[f * 3], py = a.cl_centroid[f * 3 + 1], pz = a.cl_centroid[f * 3 + 2];
            if (threadIdx.x == 0) s_flag_any = 0;
            __syncthreads();
            bool close = false;
            for (int t = threadIdx.x; t < n_mo; t += kSingle) {
                const double dx = (double)__fsub_rn(px, mo_centroid[t * 3]), dy = (double)__fsub_rn(py, mo_centroid[t * 3 + 1]),
                             dz = (double)__fsub_rn(pz, mo_centroid[t * 3 + 2]);
                const double dist = sqrt(dx * dx + dy * dy + dz * dz);
                close |= dist < (double)a.catch_up;
            }
            if (close) s_flag_any = 1;
            __syncthreads();
            const bool any = s_flag_any != 0;
            if (!any) {
                if (n_mo < a.momax) {
                    if (threadIdx.x == 0) {
                        mo_centroid[n_mo * 3] = px; mo_centroid[n_mo * 3 + 1] = py; mo_centroid[n_mo * 3 + 2] = pz;
                        mo_conf[n_mo] = a.static_confidence + 1;  // MovingObjectCentroid ctor, .h:91
                    }
                    n_mo++;
                } else if (threadIdx.x == 0) {
                    atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_MOVING_CAP);
                }
            }
            __syncthreads();
        }
    }
    MOR_TRACE(27);
    if (threadIdx.x == 0) {
        if (res_count >= a.moving_confidence) {  // pop_front both deques, cpp:511-512
            ts->corr_head = (corr_head + 1) % D; ts->corr_count = corr_count - 1;
            ts->res_head = (res_head + 1) % D; ts->res_count = res_count - 1;
        } else {
            ts->corr_count = corr_count; ts->res_count = res_count; ts->res_head = res_head % D;
        }
        ts->n_mo[a.mo_parity] = n_mo;
    }
}

// The clustering grid and the scan states go back to "all zero" for the next frame (in the last phase, beside the
// compaction: nothing reads them any more).
__device__ __forceinline__ void frame_cleanup(const FramePtrs& a, int cta, int G) {
    const int n_cells = frame_vars().n_cells;
    for (int i = cta * kT + threadIdx.x; i < n_cells; i += G * kT)
        *reinterpret_cast<uint4*>(a.table + a.cell_list[i]) = make_uint4(0u, 0u, 0u, 0u);
    for (int t = cta * kT + threadIdx.x; t < a.tiles_pts; t += G * kT) a.st_ingest[t] = 0ull;
}
// The single-CTA end of the moving-test phase.
__device__ __forceinline__ void phase_chain_tail(const FramePtrs& a) {
    if (a.two_frames) phase_chain(a);
    __syncthreads();
    if (threadIdx.x == 0) a.counts[MOR_CNT_NMO] = a.track->n_mo[a.mo_parity];
}

// ===================================================================================== phase K: filterCloud
// filterCloud (cpp:613-696).
//  Tracking part (cpp:630-671): 1-NN of every confirmed mover among the current centroids, unconditional selection of
//  that cluster (cpp:644-648), confidence update and erase. It is tiny (|mo_vec| x K distance evaluations), so EVERY
//  CTA recomputes the selection into shared memory; one CTA alone (`writer`) writes the updated mo_vec into the other
//  half of a double buffer - the host makes it current when filterCloud is called, so the phase can run at the end of
//  the frame kernel (a frame that is never filtered leaves mo_vec untouched, as in the reference).
//  Output part: ExtractIndices(negative) of the moving points + append of the ground points (cpp:673-684), written as
//  pcl::PointXYZI wire records (cpp:690); stable single-pass compaction over [cloud | ground].
constexpr int kOutTile = kT;
constexpr int kRemovedBits = kSmallK;  // a frame with more clusters takes the LARGE filter

struct FilterShared {
    unsigned removed[kRemovedBits / 32];
    int total, keep_base;
    int nn_k[kT]; float nn_d[kT];  // nearest cluster of one chunk of mo_vec entries
};

// LARGE (K > kRemovedBits): marker_cluster already holds every entry's nearest cluster and cluster_removed the removal
// set (filter_markers_large, filter_mark_large); the distance is recomputed from the two centroids (the same sqdist3 as
// the search: the same float).
template <bool LARGE = false>
__device__ __forceinline__ int filter_tracking(const FramePtrs& a, FilterShared& sh, bool writer) {
    const int mo_parity = a.mo_parity;
    const int K = a.counts[MOR_CNT_K];
    const int nc = frame_vars().nc;
    TrackState* ts = a.track;
    const int n_mo = ts->n_mo[mo_parity];
    const float* mo_c_in = a.mo_centroid + (size_t)mo_parity * a.momax * 3;
    const int* mo_f_in = a.mo_conf + (size_t)mo_parity * a.momax;
    float* mo_c_out = a.mo_centroid + (size_t)(mo_parity ^ 1) * a.momax * 3;
    int* mo_f_out = a.mo_conf + (size_t)(mo_parity ^ 1) * a.momax;
    __syncthreads();
    if (threadIdx.x == 0) { sh.total = 0; sh.keep_base = 0; }
    if (!LARGE)
        for (int t = threadIdx.x; t < (K + 31) / 32; t += kT) sh.removed[t] = 0u;
    __syncthreads();
    // K == 0: un-built kd-tree in the reference (UB) -> entries untouched
    for (int base = 0; base < n_mo && K > 0; base += kT) {
        if (!LARGE) {   // a warp per entry
            const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
            for (int u = warp; u < kT && base + u < n_mo; u += kWarps) {
                const int e = base + u;
                float d;
                const int k = nn_warp(a.cl_centroid, K, mo_c_in[e * 3], mo_c_in[e * 3 + 1], mo_c_in[e * 3 + 2], &d, lane);
                if (lane == 0) { sh.nn_k[u] = k; sh.nn_d[u] = d; }
            }
        }
        __syncthreads();
        const int t = base + threadIdx.x;
        bool keep = false;
        float cx = 0, cy = 0, cz = 0; int conf = 0;
        if (t < n_mo) {
            cx = mo_c_in[t * 3]; cy = mo_c_in[t * 3 + 1]; cz = mo_c_in[t * 3 + 2];
            conf = mo_f_in[t];
            float d;
            int k;
            if (LARGE) {
                k = __ldcg(&a.marker_cluster[t]);
                d = sqdist3(cx, cy, cz, __ldcg(&a.cl_centroid[k * 3]), __ldcg(&a.cl_centroid[k * 3 + 1]), __ldcg(&a.cl_centroid[k * 3 + 2]));
            } else {
                d = sh.nn_d[threadIdx.x];
                k = sh.nn_k[threadIdx.x];
                if (writer) a.marker_cluster[t] = k;
                atomicOr(&sh.removed[k >> 5], 1u << (k & 31));
            }
            atomicAdd(&sh.total, a.cl_size[k]);
            if (!a.cl_flags[k] || d > a.leave_off) {  // cpp:650
                conf--;
                keep = conf != 0;
            } else {
                cx = a.cl_centroid[k * 3]; cy = a.cl_centroid[k * 3 + 1]; cz = a.cl_centroid[k * 3 + 2];
                if (conf < a.static_confidence + 1) conf++;
                keep = true;
            }
        }
        if (writer) {  // ordered erase (cpp:655-660): survivors keep their relative order
            int tot;
            const int r = block_exclusive_scan<int, kT>(keep ? 1 : 0, &tot);
            if (keep) {
                const int o = sh.keep_base + r;
                mo_c_out[o * 3] = cx; mo_c_out[o * 3 + 1] = cy; mo_c_out[o * 3 + 2] = cz;
                mo_f_out[o] = conf;
            }
            __syncthreads();
            if (threadIdx.x == 0) sh.keep_base += tot;
        }
        __syncthreads();
    }
    __syncthreads();
    const int overflow = sh.total > nc ? 1 : 0;  // ExtractIndices: more indices than points => error, empty output (A18)
    if (writer) {
        if (K == 0) {  // entries untouched: copy through
            for (int t = threadIdx.x; t < n_mo; t += kT) {
                mo_c_out[t * 3] = mo_c_in[t * 3]; mo_c_out[t * 3 + 1] = mo_c_in[t * 3 + 1]; mo_c_out[t * 3 + 2] = mo_c_in[t * 3 + 2];
                mo_f_out[t] = mo_f_in[t];
            }
        }
        if (!LARGE)
            for (int k = threadIdx.x; k < K; k += kT) a.cluster_removed[k] = (sh.removed[k >> 5] >> (k & 31)) & 1u;
        if (threadIdx.x == 0) {
            const int kept = K > 0 ? sh.keep_base : n_mo;
            ts->n_mo[mo_parity ^ 1] = kept;  // the host flips the parity when filterCloud commits the frame
            ts->extract_overflow = overflow;
            ts->n_markers = K > 0 ? n_mo : 0;
            a.counts[CNT_SPEC_NMO] = kept;
            a.counts[CNT_SPEC_OVERFLOW] = overflow;
        }
    }
    return overflow;
}

// The LARGE filter's group-wide steps, each followed by a group barrier (k_filter_again: a launch each). 1: the nearest
// current cluster of every mo_vec entry (chunks of entries dealt out over the CTAs) and an empty removal set.
__device__ __forceinline__ void filter_markers_large(const FramePtrs& a, int cta, int G, float4* tile) {
    const int K = __ldcg(&a.counts[MOR_CNT_K]);
    const int n_mo = __ldcg(&a.track->n_mo[a.mo_parity]);
    const float* mo_c_in = a.mo_centroid + (size_t)a.mo_parity * a.momax * 3;
    for (int k = cta * kT + threadIdx.x; k < K; k += G * kT) a.cluster_removed[k] = 0;
    for (int c = cta; c * kNnQ < n_mo; c += G) nn_chunk(mo_c_in, c * kNnQ, min(kNnQ, n_mo - c * kNnQ), a.cl_centroid, K, tile, a.marker_cluster, nullptr);
}
// 2: the clusters selected by the entries are removed (cpp:644-648).
__device__ __forceinline__ void filter_mark_large(const FramePtrs& a, int cta, int G) {
    const int n_mo = __ldcg(&a.track->n_mo[a.mo_parity]);
    for (int e = cta * kT + threadIdx.x; e < n_mo; e += G * kT) {
        const int k = __ldcg(&a.marker_cluster[e]);
        if (k >= 0) a.cluster_removed[k] = 1;  // (-1: no centroid compared below FLT_MAX)
    }
}

struct FilterTileIn { float4 p; int c; };  // a thread's item of a tile: the point and, for a cloud point, its cluster
__device__ __forceinline__ FilterTileIn filter_tile_load(const FramePtrs& a, int tile) {
    const int nc = frame_vars().nc, ng = frame_vars().ng;
    const int t = tile * kOutTile + threadIdx.x;
    FilterTileIn in;
    in.p = make_float4(0, 0, 0, 0); in.c = -1;
    if (t < nc) { in.p = a.pts[t]; in.c = a.cid[t]; }
    else if (t < nc + ng) in.p = a.gpts[t - nc];
    return in;
}
__device__ __forceinline__ bool cluster_is_removed(const FramePtrs& a, const FilterShared& sh, int c, bool large) {
    return large ? __ldcg(&a.cluster_removed[c]) != 0 : ((sh.removed[c >> 5] >> (c & 31)) & 1u) != 0;
}
template <bool LARGE = false>
__device__ __forceinline__ void filter_tile(const FramePtrs& a, const FilterShared& sh, int overflow, int tile, int last_tile, const FilterTileIn& in) {
    const int nc = frame_vars().nc, ng = frame_vars().ng;
    const int t = tile * kOutTile + threadIdx.x;
    bool keep = false;
    const float4 p = in.p;
    if (t < nc) {
        const int c = in.c;
        const bool removed = overflow || (c >= 0 && cluster_is_removed(a, sh, c, LARGE));
        keep = !removed;
        if (removed) a.removed_mask[a.cloud_src[t]] = 2;
    } else if (t < nc + ng) {
        keep = true;
    }
    int tot;
    const int in_block = block_exclusive_scan<int, kT>(keep ? 1 : 0, &tot);
    const int before = (int)tile_prefix_wide<kT>(a.st_out, tile, (unsigned long long)tot);
    if (keep) {
        const int o = before + in_block;
        a.out[2 * o] = make_float4(p.x, p.y, p.z, 1.0f);
        a.out[2 * o + 1] = make_float4(p.w, 0.f, 0.f, 0.f);
    }
    if (tile == last_tile && threadIdx.x == 0) a.counts[CNT_SPEC_NOUT] = before + tot;
}

// The same tile with four consecutive items per thread (4096 per CTA and round): for groups that have several rounds of
// tiles per CTA (the back half of a pipelined launch on 23 CTAs, a sequence of a batch on 4) - a quarter of the rounds, each
// a chain of scan, prefix round trip and stores.
constexpr int kOutWide = 4;
template <bool LARGE = false>
__device__ __forceinline__ void filter_tile_wide(const FramePtrs& a, const FilterShared& sh, int overflow, int tile, int last_tile) {
    const int nc = frame_vars().nc, ng = frame_vars().ng;
    const int t0 = (tile * kOutTile + (int)threadIdx.x) * kOutWide;
    float4 p[kOutWide];
    bool keep[kOutWide];
    int cnt = 0;
#pragma unroll
    for (int q = 0; q < kOutWide; q++) {
        const int t = t0 + q;
        keep[q] = false;
        p[q] = make_float4(0, 0, 0, 0);
        if (t < nc) {
            p[q] = a.pts[t];
            const int c = a.cid[t];
            const bool removed = overflow || (c >= 0 && cluster_is_removed(a, sh, c, LARGE));
            keep[q] = !removed;
            if (removed) a.removed_mask[a.cloud_src[t]] = 2;
        } else if (t < nc + ng) {
            p[q] = a.gpts[t - nc];
            keep[q] = true;
        }
        cnt += keep[q] ? 1 : 0;
    }
    int tot;
    const int in_block = block_exclusive_scan<int, kT>(cnt, &tot);
    const int before = (int)tile_prefix_wide<kT>(a.st_out, tile, (unsigned long long)tot);
    int o = before + in_block;
#pragma unroll
    for (int q = 0; q < kOutWide; q++) {
        if (!keep[q]) continue;
        a.out[2 * o] = make_float4(p[q].x, p[q].y, p[q].z, 1.0f);
        a.out[2 * o + 1] = make_float4(p[q].w, 0.f, 0.f, 0.f);
        o++;
    }
    if (tile == last_tile && threadIdx.x == 0) a.counts[CNT_SPEC_NOUT] = before + tot;
}

template <bool LARGE>
__device__ __forceinline__ void phase_filter_tiles(const FramePtrs& a, int cta, int G, FilterShared& sh) {
    const int total_items = frame_vars().nc + frame_vars().ng;
    if ((long long)total_items > 2ll * G * kOutTile) {  // several rounds per CTA: four items per thread
        const int last_wide = (total_items - 1) / (kOutTile * kOutWide);
        if (cta > last_wide) return;
        const int overflow = filter_tracking<LARGE>(a, sh, cta == 0);
        for (int tile = cta; tile <= last_wide; tile += G) filter_tile_wide<LARGE>(a, sh, overflow, tile, last_wide);
        return;
    }
    const int last_tile = total_items ? (total_items - 1) / kOutTile : 0;
    if (cta > last_tile) return;  // nothing to compact here (CTA 0 always has tile 0: it owns the mo_vec update)
    FilterTileIn in = filter_tile_load(a, cta);  // the first tile's loads are in flight while the tracking part runs
    const int overflow = filter_tracking<LARGE>(a, sh, cta == 0);
    for (int tile = cta; tile <= last_tile; tile += G) {
        if (tile != cta) in = filter_tile_load(a, tile);
        filter_tile<LARGE>(a, sh, overflow, tile, last_tile, in);
    }
}
// (out of line: the frame kernels run at their register limit, and the rare large-K steps should not add to it)
__device__ __noinline__ void phase_filter_large(const FramePtrs& a, int cta, int G, FilterShared& sh, unsigned long long* dyn, GroupBarrier& bar) {
    filter_markers_large(a, cta, G, reinterpret_cast<float4*>(dyn));
    bar.sync();
    filter_mark_large(a, cta, G);
    bar.sync();
    phase_filter_tiles<true>(a, cta, G, sh);
}
// Every CTA must call (the LARGE filter has group barriers in front of the tiles); K is final since the match.
template <bool LK>
__device__ __forceinline__ void phase_filter(const FramePtrs& a, int cta, int G, FilterShared& sh, unsigned long long* dyn, GroupBarrier& bar, bool cleanup = true) {
    if (cleanup) frame_cleanup(a, cta, G);
    if (LK && __ldcg(&a.counts[MOR_CNT_K]) > kRemovedBits) {
        phase_filter_large(a, cta, G, sh, dyn, bar);
    } else {
        phase_filter_tiles<false>(a, cta, G, sh);
    }
}

// Last CTA out: every counter of the frame back to zero.
template <bool LK>
__device__ __forceinline__ void frame_epilogue(const FramePtrs& a, int G) {
    __shared__ int s_last;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(&a.scratch->blocks_done, 1) == G - 1;
        __threadfence();
    }
    __syncthreads();
    if (!s_last) return;
    for (int t = threadIdx.x; t < a.tiles_pts; t += kT) a.st_out[t] = 0ull;
    if (threadIdx.x == 0) {
        Scratch* sc = a.scratch;
        sc->bar = 0u; sc->blocks_done = 0; sc->n_cells = 0; sc->n_roots = 0; sc->n_light = 0; sc->n_heavy = 0; sc->n_sorted = 0; sc->tail_match = 0u; sc->tail_chain = 0u; sc->err_early = 0;
        if (LK) sc->n_sel = 0;
        sc->ticket_ingest = 0; sc->ticket_cells = 0;  // voxel ground modes (k_ground_partition leaves its tile tickets behind)
        for (int q = 0; q < 3; q++) { sc->box_inv_min[q] = 0u; sc->box_max[q] = 0u; }
    }
}

// ===================================================================================== the frame kernel
enum Phase { PH_INGEST = 0, PH_CELLS, PH_LINK, PH_TEST, PH_JUMP, PH_CROSS, PH_ROOTS, PH_SELECT, PH_STATS, PH_MOVING, PH_FILTER, PH__COUNT };

template <int PH, bool LK>
__device__ __forceinline__ void run_phase(const FramePtrs& a, int cta, int G, FilterShared& sh, unsigned long long* dyn, GroupBarrier& bar) {
    if (PH == PH_INGEST) { if (a.skip_ingest) phase_bin_cloud(a, cta, G); else phase_ingest(a, cta, G); }
    if (PH == PH_CELLS) phase_cells(a, cta, G);
    if (PH == PH_LINK) phase_link(a, cta, G, dyn);
    if (PH == PH_TEST) phase_test(a, cta, G);
    if (PH == PH_JUMP) phase_jump(a, cta, G);
    if (PH == PH_CROSS) phase_cross(a, cta, G);
    if (PH == PH_ROOTS) phase_roots(a, cta, G);
    if (PH == PH_SELECT) {
        if (select_large<LK>(a)) {
            phase_select_large(a, cta, G, dyn, bar);
            if (a.two_frames) { int lo, hi; cta_slice(a.p_counts[MOR_CNT_NC], cta, G, &lo, &hi); transform_range<LK>(a, lo, hi); }
        } else {
            if (cta == 0) phase_select(a, dyn);
            phase_transform<LK>(a, cta, G);
        }
    }
    if (PH == PH_STATS) {
        phase_stats(a, cta, G);
        if (match_large<LK>(a)) { bar.sync(); phase_match_large(a, cta, G, dyn, bar); }
        else if (group_last_arrival(&a.scratch->tail_match, (unsigned)G)) phase_match(a, dyn);
    }
    if (PH == PH_MOVING) {
        if (a.two_frames) { if (a.method == 2) phase_lattice_count<LK>(a, cta, G); else phase_pde_count(a, cta, G); }
        if (group_last_arrival(&a.scratch->tail_chain, (unsigned)G)) phase_chain_tail(a);
    }
    if (PH == PH_FILTER) phase_filter<LK>(a, cta, G, sh, dyn, bar);
}


template <int PH, bool LK>
__device__ __forceinline__ void frame_step(const FramePtrs& a, int cta, int G, FilterShared& sh, unsigned long long* dyn, GroupBarrier& bar) {
    run_phase<PH, LK>(a, cta, G, sh, dyn, bar);
#ifdef MOR_CTA_TRACE
    __syncthreads();
    if (threadIdx.x == 0 && cta < 256) a.cta_trace[PH * 256 + cta] = global_ns();
#endif
    if (PH != PH_FILTER) bar.sync();
    if (cta == 0 && threadIdx.x == 0) a.phase_ts[PH + 1] = global_ns();  // a dozen stores per frame: the frame's own timeline
}

template <bool LK>
__device__ __forceinline__ void frame_body(const FramePtrs& a, int cta, int G, FilterShared& sh, unsigned long long* dyn) {
    GroupBarrier bar{&a.scratch->bar, 0u, (unsigned)G};
    if (cta == 0 && threadIdx.x == 0) a.phase_ts[0] = global_ns();
    frame_step<PH_INGEST, LK>(a, cta, G, sh, dyn, bar);
    load_frame_vars(a);
    frame_step<PH_CELLS, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_LINK, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_TEST, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_JUMP, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_CROSS, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_ROOTS, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_SELECT, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_STATS, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_MOVING, LK>(a, cta, G, sh, dyn, bar);
    frame_step<PH_FILTER, LK>(a, cta, G, sh, dyn, bar);
    frame_epilogue<LK>(a, G);
}

// ===================================================================================== pipelined launch
// Throughput mode (mor_set_pipelining; frames are known one ahead - replay, the streaming calls): clustering a frame needs
// nothing of the frame before it, so ONE launch runs the front half of frame f+1 (ingest ... cluster selection) on the
// first Gf CTAs beside the back half of frame f (cluster statistics, transform, match, moving test, chain, filter) on the
// others. The two groups have their own barriers and counters and touch disjoint state: what the back half reads of
// frame f and f-1 is triple-buffered (points, sorted points, cluster ids, cluster tables, counts) or double-buffered by
// frame parity (ground points, source indices, masks, the clusters' coordinate sums and boxes, and what the statistics
// phase resolves each point's cluster from: slead, hook, rmin, cid_of_pos; scid, which it writes) on the host side
// (mor_b200.cu, fill_frame). The front half's other per-frame arrays (cells, pair lists, rsize, root_list, cid_of_root)
// are read by no back half.
// Four instantiations of the same two bodies, picked per handle by mor_b200.cu (pipe_variant):
//  - k_frame_pipe: crop ground mode, method 2.
//  - k_frame_pipe_ground (GROUND): voxel ground modes. Frame f+1's nine ground launches (mor_ground.cuh) run on the stream
//    before this launch, i.e. after the launch that ran f's front half and before f's back half. What they write, against
//    what the back half of f reads later:
//      k_ingest_raw: counts of f+1 (zeroed and filled by its last tile; a slot of the triple-buffered counts, f's slot is
//        another), track->frames (read by the ingest alone), point_class (per point; read by the front half and the taps of
//        the current frame, never by a back half), removed_mask (parity of f+1; f's filter marks the other parity), the
//        Scratch box words and ticket_ingest, st_ingest, bin_hist, rpts / rsrc / is_ground (ground stage only);
//      k_ground_keys / k_scan_cells / k_ground_scatter: the dense cell_count / cell_start / cell_key / skey tables, vkey,
//        vox_count, ggrid / vdesc, st_cells, ticket_cells (ground stage only), spts (f+1's slot of three), ERRFLAGS in
//        the counts of f+1;
//      k_scan_voxels / k_voxel_eval / k_ground_mode / k_ground_mark: vox_* , vacc, bin_hist, gstate, the scan states and
//        Scratch tickets and box words they reset (ground stage only);
//      k_ground_partition: point_class, pts (slot of f+1), cloud_src / gpts / gsrc (parity of f+1), counts of f+1.
//    None of these is read by the back half of f (it reads f's and f-1's slots, f's parity, the tracking state, st_out
//    and its own Scratch words), so f's back half sees what it would have seen without the ground stage in between. The
//    front half starts at the binning (phase_bin_cloud, no housekeeping: the back half does that) and gives back the
//    ticket that k_ground_partition leaves drawn.
//  - k_frame_pipe_pde (PDE): method 1. Its moving test searches frame f's clustering grid in the back half, so a method-1
//    handle keeps the grid (table, cell_list) per frame parity; the front half leaves it standing and hands its cell
//    count over in counts[CNT_PIPE_CELLS]; the back half empties it after the search.
//  - k_frame_pipe_ground_pde: both.
// Timeline of a pipelined launch in the spare words of phase_ts (after frame_body's PH__COUNT + 1): CTA 0 of each half
// stamps its start and every barrier it passes, the last CTA out of each half stamps the end (tools/quick_bench.py,
// QB_PIPE=1). Front: start, ingest, cells, link, test, jump, cross, roots + select, end. Back: start, housekeeping,
// statistics + transform + match, moving test + chain, filter (end).
enum { TS_FRONT = PH__COUNT + 1, TS_BACK = TS_FRONT + 9 };
static_assert(TS_BACK + 5 <= 32, "phase_ts holds 32 words");
__device__ __forceinline__ void pipe_stamp(const FramePtrs& a, int cta, int word) {
    if (cta == 0 && threadIdx.x == 0) a.phase_ts[word] = global_ns();
}

template <bool GROUND, bool PDE, bool LK>
__device__ __forceinline__ void front_body(const FramePtrs& a, int cta, int G, unsigned long long* dyn) {
    GroupBarrier bar{&a.scratch->bar, 0u, (unsigned)G};
    pipe_stamp(a, cta, TS_FRONT);
    if (GROUND) phase_bin_cloud(a, cta, G, /*housekeep=*/false);
    else phase_ingest(a, cta, G, /*housekeep=*/false);
    bar.sync(); pipe_stamp(a, cta, TS_FRONT + 1);
    load_frame_vars(a);
    phase_cells(a, cta, G); bar.sync(); pipe_stamp(a, cta, TS_FRONT + 2);
    phase_link(a, cta, G, dyn); bar.sync(); pipe_stamp(a, cta, TS_FRONT + 3);
    phase_test(a, cta, G); bar.sync(); pipe_stamp(a, cta, TS_FRONT + 4);
    phase_jump(a, cta, G); bar.sync(); pipe_stamp(a, cta, TS_FRONT + 5);
    phase_cross(a, cta, G); bar.sync(); pipe_stamp(a, cta, TS_FRONT + 6);
    phase_roots(a, cta, G);
    // (the last CTA in selects the clusters: no barrier in front of it; a large-K frame is selected by the whole group)
    if (group_last_arrival(&a.scratch->tail_centroids, (unsigned)G) && !select_large<LK>(a)) phase_select(a, dyn);
    bar.sync();
    if (select_large<LK>(a)) { phase_select_large(a, cta, G, dyn, bar); bar.sync(); }
    pipe_stamp(a, cta, TS_FRONT + 7);
    if (PDE) {  // the grid stays for the back half's search: only the scan states go back to zero here
        for (int t = cta * kT + threadIdx.x; t < a.tiles_pts; t += G * kT) a.st_ingest[t] = 0ull;
        if (cta == 0 && threadIdx.x == 0) a.counts[CNT_PIPE_CELLS] = frame_vars().n_cells;
    } else {
        frame_cleanup(a, cta, G);
    }
    // last CTA of the group out: the front half's counters back to zero
    __shared__ int s_last_front;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last_front = atomicAdd(&a.scratch->blocks_done, 1) == G - 1;
        __threadfence();
    }
    __syncthreads();
    if (s_last_front && threadIdx.x == 0) {
        a.phase_ts[TS_FRONT + 8] = global_ns();
        Scratch* sc = a.scratch;
        sc->bar = 0u; sc->blocks_done = 0; sc->n_cells = 0; sc->n_roots = 0; sc->n_light = 0; sc->n_heavy = 0; sc->n_sorted = 0; sc->tail_centroids = 0u;
        sc->err_early = 0;
        if (LK) sc->n_sel = 0;
        if (GROUND) sc->ticket_ingest = 0;  // (drawn by k_ground_partition; frame_epilogue resets it in one kernel per frame)
    }
}

// (GROUND does not change the back half; it keeps every kernel's instantiations of the two bodies its own, so that their
// static shared variables stay local to one kernel and k_frame_pipe's shared layout is what it was before the variants)
template <bool GROUND, bool PDE, bool LK>
__device__ __forceinline__ void back_body(const FramePtrs& a, int cta, int G, FilterShared& sh, unsigned long long* dyn) {
    GroupBarrier bar{&a.scratch->bar_back, 0u, (unsigned)G};
    if (threadIdx.x == 0) {  // (the cell count belongs to the front half, which is busy with the next frame)
        FrameVars& v = frame_vars();
        v.n_cells = 0; v.nc = __ldcg(&a.counts[MOR_CNT_NC]); v.ng = __ldcg(&a.counts[MOR_CNT_NG]);
    }
    __syncthreads();
    pipe_stamp(a, cta, TS_BACK);
    frame_housekeeping(a, cta, G);
    bar.sync(); pipe_stamp(a, cta, TS_BACK + 1);
    stats_transform<LK>(a, cta, G);
    if (match_large<LK>(a)) { bar.sync(); phase_match_large(a, cta, G, dyn, bar); }
    else if (group_last_arrival(&a.scratch->tail_match_back, (unsigned)G)) phase_match(a, dyn);
    bar.sync(); pipe_stamp(a, cta, TS_BACK + 2);
    if (a.two_frames) { if (PDE) phase_pde_count(a, cta, G); else phase_lattice_count<LK>(a, cta, G); }
    if (group_last_arrival(&a.scratch->tail_chain, (unsigned)G)) phase_chain_tail(a);
    bar.sync(); pipe_stamp(a, cta, TS_BACK + 3);
    if (PDE) {  // the search is over: this frame's clustering grid goes back to "all zero" (frame_cleanup's first loop)
        const int n_cells = a.counts[CNT_PIPE_CELLS];
        for (int i = cta * kT + threadIdx.x; i < n_cells; i += G * kT)
            *reinterpret_cast<uint4*>(a.table + a.cell_list[i]) = make_uint4(0u, 0u, 0u, 0u);
    }
    phase_filter<LK>(a, cta, G, sh, dyn, bar, /*cleanup=*/false);
    __shared__ int s_last_back;
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last_back = atomicAdd(&a.scratch->blocks_done_back, 1) == G - 1;
        __threadfence();
    }
    __syncthreads();
    if (!s_last_back) return;
    for (int t = threadIdx.x; t < a.tiles_pts; t += kT) a.st_out[t] = 0ull;
    if (threadIdx.x == 0) {
        a.phase_ts[TS_BACK + 4] = global_ns();
        Scratch* sc = a.scratch;
        sc->bar_back = 0u; sc->blocks_done_back = 0; sc->tail_match_back = 0u; sc->tail_chain = 0u;
    }
}

// Every frame kernel below is a template on LK ("large-K"): the instantiation with LK = true serves handles whose
// max_clusters exceeds kSmallK and carries the group-wide steps for frames with more clusters; LK = false is the code of
// every other handle, with no trace of them (mor_b200.cu picks the instantiation per handle).
//
// Front half of `f` on the CTAs [0, Gf), back half of `b` on the rest; Gf = gridDim.x: front only, Gf = 0: back only.
template <bool GROUND, bool PDE, bool LK>
__device__ __forceinline__ void frame_pipe_variant(const FramePtrs& f, const FramePtrs& b, int Gf) {
    extern __shared__ __align__(128) unsigned long long dyn[];
    __shared__ FilterShared sh;
    if ((int)blockIdx.x < Gf) front_body<GROUND, PDE, LK>(f, blockIdx.x, Gf, dyn);
    else back_body<GROUND, PDE, LK>(b, (int)blockIdx.x - Gf, (int)gridDim.x - Gf, sh, dyn);
}
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame_pipe(const __grid_constant__ FramePtrs f, const __grid_constant__ FramePtrs b, int Gf) {
    frame_pipe_variant<false, false, LK>(f, b, Gf);
}
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame_pipe_ground(const __grid_constant__ FramePtrs f, const __grid_constant__ FramePtrs b, int Gf) {
    frame_pipe_variant<true, false, LK>(f, b, Gf);
}
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame_pipe_pde(const __grid_constant__ FramePtrs f, const __grid_constant__ FramePtrs b, int Gf) {
    frame_pipe_variant<false, true, LK>(f, b, Gf);
}
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame_pipe_ground_pde(const __grid_constant__ FramePtrs f, const __grid_constant__ FramePtrs b, int Gf) {
    frame_pipe_variant<true, true, LK>(f, b, Gf);
}

// One sequence, the whole grid is its group; the frame's arguments travel in the constant bank.
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame(const __grid_constant__ FramePtrs a) {
    extern __shared__ __align__(128) unsigned long long dyn[];
    __shared__ FilterShared sh;
    frame_body<LK>(a, blockIdx.x, gridDim.x, sh, dyn);
}

// S sequences per launch: grid = groups x G CTAs; group g steps sequences g, g + groups, ... (each through all
// phases, independently of the other groups), G CTAs per sequence.
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame_batch(const FramePtrs* __restrict__ P, int S, int G) {
    extern __shared__ __align__(128) unsigned long long dyn[];
    __shared__ FilterShared sh;
    const int group = blockIdx.x / G, cta = blockIdx.x % G, groups = gridDim.x / G;
    for (int seq = group; seq < S; seq += groups) frame_body<LK>(P[seq], cta, G, sh, dyn);
}

// One phase per launch (per-phase timing; the kernel boundary is the barrier). Same grid, same striding.
template <int PH, bool LK>
__global__ void __launch_bounds__(kT, 1) k_phase(const __grid_constant__ FramePtrs a) {
    extern __shared__ __align__(128) unsigned long long dyn[];
    __shared__ FilterShared sh;
    GroupBarrier bar{&a.scratch->bar, 0u, gridDim.x};  // (the large-K steps of select, match and filter)
    if (PH != PH_INGEST) load_frame_vars(a);
    run_phase<PH, LK>(a, blockIdx.x, gridDim.x, sh, dyn, bar);
    if (PH == PH_FILTER) frame_epilogue<LK>(a, gridDim.x);
    if (LK && (PH == PH_SELECT || PH == PH_STATS)) {  // last CTA out: the barrier back to zero for the next launch
        __shared__ int s_last;
        __syncthreads();
        if (threadIdx.x == 0) s_last = atomicAdd(&a.scratch->blocks_done, 1) == (int)gridDim.x - 1;
        __syncthreads();
        if (s_last && threadIdx.x == 0) { a.scratch->bar = 0u; a.scratch->blocks_done = 0; }
    }
}

// filterCloud called again on a frame that was already filtered (the reference then runs the tracking update once
// more on the updated mo_vec): the filter phase alone. Tiles by ticket, so a plain launch suffices. A frame with more
// than kRemovedBits clusters has its markers and removal set made first by k_filter_markers and k_filter_mark (launched
// in front of it by handles whose kmax allows such frames; they do nothing for a smaller frame).
__global__ void __launch_bounds__(kT, 1) k_filter_markers(const __grid_constant__ FramePtrs a) {
    extern __shared__ __align__(128) unsigned long long dyn[];
    if (__ldcg(&a.counts[MOR_CNT_K]) > kRemovedBits) filter_markers_large(a, blockIdx.x, gridDim.x, reinterpret_cast<float4*>(dyn));
}
__global__ void __launch_bounds__(kT, 1) k_filter_mark(const __grid_constant__ FramePtrs a) {
    if (__ldcg(&a.counts[MOR_CNT_K]) > kRemovedBits) filter_mark_large(a, blockIdx.x, gridDim.x);
}
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_filter_again(const __grid_constant__ FramePtrs a) {
    __shared__ FilterShared sh;
    __shared__ int s_tile, s_last;
    if (threadIdx.x == 0) s_tile = atomicAdd(&a.scratch->ticket_out, 1);
    load_frame_vars(a);
    const int tile = s_tile;
    const int total_items = frame_vars().nc + frame_vars().ng;
    const int last_tile = total_items ? (total_items - 1) / kOutTile : 0;
    if (tile <= last_tile) {
        const FilterTileIn in = filter_tile_load(a, tile);
        if (LK && __ldcg(&a.counts[MOR_CNT_K]) > kRemovedBits) {
            const int overflow = filter_tracking<true>(a, sh, tile == 0);
            filter_tile<true>(a, sh, overflow, tile, last_tile, in);
        } else {
            const int overflow = filter_tracking(a, sh, tile == 0);
            filter_tile(a, sh, overflow, tile, last_tile, in);
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) s_last = atomicAdd(&a.scratch->out_blocks_done, 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (s_last) {
        for (int t = threadIdx.x; t < a.tiles_pts; t += kT) a.st_out[t] = 0ull;
        if (threadIdx.x == 0) { a.scratch->ticket_out = 0; a.scratch->out_blocks_done = 0; }
    }
}

}  // namespace mor
