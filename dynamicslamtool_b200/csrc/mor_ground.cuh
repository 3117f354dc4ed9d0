// mor_ground.cuh — voxel-covariance ground removal (ground_mode 1 and 2), the path that is dead and
// crashing in the reference (groundPlaneRemoval(x,y), src/MovingObjectRemoval.cpp:90-200, call commented
// out at :527). Semantics = the repaired restatement in oracle/mor_oracle.cpp (DESIGN.md §8):
//   trim (A1) -> VoxelGrid(gp_leaf) centroids (A14) -> ball query r = gp_leaf over raw_cloud (A6, strict)
//   -> per-ball scatter matrix -> mode 1: |S_xz|,|S_yz|,|S_zz| < 0.001 (cpp:145), Z bin (cpp:166)
//                               mode 2: closed-form symmetric eigen-solve, planarity + normal test, bin
//                                       along the voxel's own normal
//   -> histogram of bins, mode bin (mode 2: every bin >= 25 % of it) -> ground = union of the balls of the
//   accepted voxels in the selected bins -> stable partition of raw_cloud into cloud / gp_indices.
// Stages: radix-free counting sort on a dense voxel key, exact fixed-point voxel sums, one thread per
// voxel for the 27-cell ball statistics (double moments relative to the voxel centroid).
#pragma once
#include "mor_kernels.cuh"

namespace mor {

struct VoxDesc {  // pcl::VoxelGrid index space: idx = i + j*dx + k*dx*dy with (i,j,k) = floor(p*inv_leaf) - min_b
    long long minb[3];
    int div[3];
    int ncells;
};

struct GroundPtrs {
    int mode;                 // MOR_GROUND_VOXEL_COV / MOR_GROUND_VOXEL_EIGEN
    float leaf, inv_leaf, r2, bin_gap, planarity, bin_width;
    double ball_cell_h;       // leaf * (1 + 2^-10)
    float4* rpts; int* rsrc;  // raw_cloud (after the x/y trim), raw -> input index
    uint8_t* is_ground;
    int* vkey;                // voxel index of every raw point
    int* vox_count; int* vox_ord; unsigned long long* st_vox;
    int* vox_n; unsigned long long* vacc; float* vox_info;
    int* bin_hist;            // 65536 bins
    GridDesc* ggrid; VoxDesc* vdesc;
    int* gstate;              // [0] ticket_vox, [1] n_vox, [2] best bin, [3] threshold count
    int tiles_vox;
};

// ===================================================================================== G1
// fromPCLPointCloud2 + PassThrough x,y (cpp:94-102): stable compaction of the in-range points into
// raw_cloud, bounding box of raw_cloud, resets of the per-frame ground state.
// `nblocks` blocks take part (one tile each): blocks_for(a.n).
__device__ __forceinline__ void ingest_raw(const FramePtrs& a, const GroundPtrs& gp, unsigned nblocks) {
    __shared__ int s_tile;
    if (threadIdx.x == 0) s_tile = atomicAdd(&a.scratch->ticket_ingest, 1);
    __syncthreads();
    const int tile = s_tile;
    const uint32_t i = (uint32_t)tile * kBlock + threadIdx.x;
    const uint32_t stride = nblocks * kBlock;
    for (uint32_t t = i; t < 65536u; t += stride) gp.bin_hist[t] = 0;
    float x = 0.f, y = 0.f, z = 0.f, w = 0.f;
    bool in = false;
    if (i < a.n) {
        const uint8_t* p = a.in + (size_t)i * a.step;
        if (a.in_mode == 0) {
            float4 v = __ldg(reinterpret_cast<const float4*>(p));
            x = v.x; y = v.y; z = v.z; w = v.w;
        } else {
            x = load_f32(p + a.off_x, a.in_mode); y = load_f32(p + a.off_y, a.in_mode); z = load_f32(p + a.off_z, a.in_mode);
            w = a.off_i != 0xFFFFFFFFu ? load_f32(p + a.off_i, a.in_mode) : 0.f;
        }
        in = isfinite(x) && isfinite(y) && isfinite(z) && !(x < -a.trim_x || x > a.trim_x) && !(y < -a.trim_y || y > a.trim_y);
        a.point_class[i] = 0;
        a.removed_mask[i] = in ? 1 : 0;
    }
    int total;
    const int in_block = block_exclusive_scan<int>(in ? 1 : 0, &total);
    const int before = (int)tile_exclusive_prefix(a.st_ingest, tile, (unsigned long long)total);
    if (in) {
        const int r = before + in_block;
        gp.rpts[r] = make_float4(x, y, z, w);
        gp.rsrc[r] = (int)i;
        gp.is_ground[r] = 0;
    }
    {
        const unsigned kx = fkey(x), ky = fkey(y), kz = fkey(z);
        const unsigned ix = __reduce_max_sync(kFull, in ? ~kx : 0u), iy = __reduce_max_sync(kFull, in ? ~ky : 0u), iz = __reduce_max_sync(kFull, in ? ~kz : 0u);
        const unsigned mx = __reduce_max_sync(kFull, in ? kx : 0u), my = __reduce_max_sync(kFull, in ? ky : 0u), mz = __reduce_max_sync(kFull, in ? kz : 0u);
        if ((threadIdx.x & 31) == 0 && (ix | mx)) {
            atomicMax(&a.scratch->box_inv_min[0], ix); atomicMax(&a.scratch->box_inv_min[1], iy); atomicMax(&a.scratch->box_inv_min[2], iz);
            atomicMax(&a.scratch->box_max[0], mx); atomicMax(&a.scratch->box_max[1], my); atomicMax(&a.scratch->box_max[2], mz);
        }
    }
    const int last_tile = a.n ? (int)((a.n - 1) / kBlock) : 0;
    if (tile == last_tile && threadIdx.x == 0) {
        int* c = a.counts;
        for (int k = 0; k < MOR_NCOUNTS; k++) c[k] = 0;
        c[MOR_CNT_N] = (int)a.n; c[MOR_CNT_NT] = before + total;
        c[MOR_CNT_TWO_FRAMES] = a.two_frames;
        if (a.two_frames) { c[MOR_CNT_KPREV] = a.p_counts[MOR_CNT_K]; c[MOR_CNT_NCPREV] = a.p_counts[MOR_CNT_NC]; }
        c[MOR_CNT_FRAME] = a.track->frames + 1;
        a.track->frames += 1;
    }
}
__global__ void __launch_bounds__(kBlock) k_ingest_raw(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    ingest_raw(a, gp, gridDim.x);
}

// ===================================================================================== G2
// Ball-query grid (cell edge leaf*(1+2^-10) over the raw bounding box) and VoxelGrid index of every raw
// point; both histograms. Every block derives the two descriptors from the reduced box.
__device__ __forceinline__ void ground_keys(const FramePtrs& a, const GroundPtrs& gp, int block) {
    __shared__ GridDesc s_g;
    __shared__ VoxDesc s_v;
    const int nraw = a.counts[MOR_CNT_NT];
    if (threadIdx.x == 0) {
        const Scratch* sc = a.scratch;
        float lo[3], hi[3];
#pragma unroll
        for (int q = 0; q < 3; q++) { lo[q] = nraw ? fkey_inv(~sc->box_inv_min[q]) : 0.f; hi[q] = nraw ? fkey_inv(sc->box_max[q]) : 0.f; }
        GridDesc g;
        const double inv_h = 1.0 / gp.ball_cell_h;
        g.ox = (double)lo[0]; g.oy = (double)lo[1]; g.oz = (double)lo[2]; g.inv_h = inv_h;
        const double fx = floor(((double)hi[0] - g.ox) * inv_h) + 1.0, fy = floor(((double)hi[1] - g.oy) * inv_h) + 1.0, fz = floor(((double)hi[2] - g.oz) * inv_h) + 1.0;
        VoxDesc v;
        double vd[3];
#pragma unroll
        for (int q = 0; q < 3; q++) {
            v.minb[q] = (long long)floorf(__fmul_rn(lo[q], gp.inv_leaf));                       // min_b = floor(min_p * inverse_leaf_size)
            vd[q] = (double)((long long)floorf(__fmul_rn(hi[q], gp.inv_leaf)) - v.minb[q] + 1);  // div_b = max_b - min_b + 1
        }
        const bool too_big = fx * fy * fz > (double)a.max_cells || vd[0] * vd[1] * vd[2] > (double)a.max_cells;
        if (too_big) { g.nx = g.ny = g.nz = 1; v.div[0] = v.div[1] = v.div[2] = 1; }
        else { g.nx = (int)fx; g.ny = (int)fy; g.nz = (int)fz; v.div[0] = (int)vd[0]; v.div[1] = (int)vd[1]; v.div[2] = (int)vd[2]; }
        g.ncells = g.nx * g.ny * g.nz;
        v.ncells = v.div[0] * v.div[1] * v.div[2];
        s_g = g; s_v = v;
        if (block == 0) {
            *gp.ggrid = g; *gp.vdesc = v;
            if (too_big) atomicOr(&a.counts[MOR_CNT_ERRFLAGS], ERR_GROUND_CAP);
        }
    }
    __syncthreads();
    const int r = block * kBlock + threadIdx.x;
    if (r >= nraw) return;
    const float4 p = gp.rpts[r];
    const GridDesc& g = s_g;
    int cx = (int)floor(((double)p.x - g.ox) * g.inv_h), cy = (int)floor(((double)p.y - g.oy) * g.inv_h), cz = (int)floor(((double)p.z - g.oz) * g.inv_h);
    cx = min(max(cx, 0), g.nx - 1); cy = min(max(cy, 0), g.ny - 1); cz = min(max(cz, 0), g.nz - 1);
    const int key = (cz * g.ny + cy) * g.nx + cx;
    a.cell_key[r] = key;
    atomicAdd(&a.cell_count[key], 1);
    const VoxDesc& v = s_v;
    long long i0 = (long long)floorf(__fmul_rn(p.x, gp.inv_leaf)) - v.minb[0];
    long long i1 = (long long)floorf(__fmul_rn(p.y, gp.inv_leaf)) - v.minb[1];
    long long i2 = (long long)floorf(__fmul_rn(p.z, gp.inv_leaf)) - v.minb[2];
    i0 = min(max(i0, 0ll), (long long)v.div[0] - 1); i1 = min(max(i1, 0ll), (long long)v.div[1] - 1); i2 = min(max(i2, 0ll), (long long)v.div[2] - 1);
    const int vk = (int)(i0 + i1 * v.div[0] + i2 * (long long)v.div[0] * v.div[1]);
    gp.vkey[r] = vk;
    atomicAdd(&gp.vox_count[vk], 1);
}
__global__ void __launch_bounds__(kBlock) k_ground_keys(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    ground_keys(a, gp, blockIdx.x);
}

// ===================================================================================== G2b
// Exclusive scan of the ball grid's per-cell histogram (counting sort of the cell keys) -> cell_start[0..ncells]. The
// histogram itself is left in place: k_ground_scatter counts it back down to zero (rank = atomicSub - 1), which both
// hands out the slots of a cell and leaves the table clean for the next frame. Persistent blocks pull tiles by ticket,
// so the launch does not depend on the (device-side) cell count.
constexpr int kScanItems = 8;
constexpr int kScanTile = kBlock * kScanItems;
__device__ __forceinline__ void scan_cells(const FramePtrs& a, int ncells) {
    __shared__ int s_tile;
    const int ntiles = (ncells + kScanTile - 1) / kScanTile;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_tile = atomicAdd(&a.scratch->ticket_cells, 1);
        __syncthreads();
        const int tile = s_tile;
        if (tile >= ntiles) return;
        const int base = tile * kScanTile + threadIdx.x * kScanItems;
        int v[kScanItems];
#pragma unroll
        for (int k = 0; k < kScanItems; k++) v[k] = (base + k < ncells) ? a.cell_count[base + k] : 0;
        int sum = 0;
#pragma unroll
        for (int k = 0; k < kScanItems; k++) sum += v[k];
        int total;
        const int in_block = block_exclusive_scan<int>(sum, &total);
        const int before = (int)tile_exclusive_prefix(a.st_cells, tile, (unsigned long long)total);
        int run = before + in_block;
#pragma unroll
        for (int k = 0; k < kScanItems; k++) {
            if (base + k < ncells) a.cell_start[base + k] = run;
            run += v[k];
        }
        if (tile == ntiles - 1 && threadIdx.x == 0) a.cell_start[ncells] = before + total;
    }
}
__global__ void __launch_bounds__(kBlock) k_scan_cells(FramePtrs a) {
    pdl_prologue();
    scan_cells(a, a.dgrid->ncells);
}

// ===================================================================================== G3
// Occupancy scan of the voxel histogram: ordinal of every occupied voxel in ascending voxel index (the
// order pcl::VoxelGrid emits its centroids in), point count per ordinal, total number of voxels.
__device__ __forceinline__ void scan_voxels(const FramePtrs& a, const GroundPtrs& gp) {
    __shared__ int s_tile;
    const int ncells = gp.vdesc->ncells;
    const int ntiles = (ncells + kTile - 1) / kTile;
    while (true) {
        __syncthreads();
        if (threadIdx.x == 0) s_tile = atomicAdd(&gp.gstate[0], 1);
        __syncthreads();
        const int tile = s_tile;
        if (tile >= ntiles) return;
        const int base = tile * kTile + threadIdx.x * kItems;
        int v[kItems];
#pragma unroll
        for (int k = 0; k < kItems; k++) v[k] = (base + k < ncells) ? gp.vox_count[base + k] : 0;
#pragma unroll
        for (int k = 0; k < kItems; k++)
            if (base + k < ncells && v[k]) gp.vox_count[base + k] = 0;
        int sum = 0;
#pragma unroll
        for (int k = 0; k < kItems; k++) sum += v[k] ? 1 : 0;
        int total;
        const int in_block = block_exclusive_scan<int>(sum, &total);
        const int before = (int)tile_exclusive_prefix(gp.st_vox, tile, (unsigned long long)total);
        int run = before + in_block;
#pragma unroll
        for (int k = 0; k < kItems; k++) {
            if (base + k < ncells && v[k]) {
                gp.vox_ord[base + k] = run; gp.vox_n[run] = v[k];
#pragma unroll
                for (int q = 0; q < 6; q++) gp.vacc[(size_t)run * 6 + q] = 0ull;
                run++;
            }
        }
        if (tile == ntiles - 1 && threadIdx.x == 0) { gp.gstate[1] = before + total; a.counts[MOR_CNT_NVOX] = before + total; }
    }
}
__global__ void __launch_bounds__(kBlock) k_scan_voxels(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    scan_voxels(a, gp);
}

// ===================================================================================== G4
// Raw points into ball-grid order; exact fixed-point coordinate sums per voxel.
__device__ __forceinline__ void ground_scatter(const FramePtrs& a, const GroundPtrs& gp, int block) {
    const int r = block * kBlock + threadIdx.x;
    const int nraw = a.counts[MOR_CNT_NT];
    if ((r & ~31) >= nraw) return;  // whole warps stay for the group reductions
    const bool in = r < nraw;
    float4 p = make_float4(0, 0, 0, 0);
    int ord = -1;
    if (in) {
        const int key = a.cell_key[r];
        const int pos = a.cell_start[key] + atomicSub(&a.cell_count[key], 1) - 1;
        p = gp.rpts[r];
        ord = gp.vox_ord[gp.vkey[r]];
        float4 sp = p;
        sp.w = __int_as_float(r);
        a.spts[pos] = sp;
        a.skey[pos] = key;
    }
    // exact voxel sums: neighbouring beams fall into the same voxel, so lanes are grouped by voxel (match.any) and
    // reduced with redux in 16/15-bit pieces before one set of 64-bit atomics per group
    const unsigned grp = __match_any_sync(kFull, ord);
    const bool leader = in && (int)(__ffs(grp) - 1) == (int)(threadIdx.x & 31);
    const float v[3] = {p.x, p.y, p.z};
#pragma unroll
    for (int q = 0; q < 3; q++) {
        long long h, l;
        split_fixed(v[q], h, l);
        const long long sh = ((long long)__reduce_add_sync(grp, (int)(h >> 16)) << 16) + (long long)__reduce_add_sync(grp, (int)(h & 0xFFFF));
        const long long sl = ((long long)__reduce_add_sync(grp, (int)(l >> 15)) << 15) + (long long)__reduce_add_sync(grp, (int)(l & 0x7FFF));
        if (leader) {
            atomicAdd(gp.vacc + (size_t)ord * 6 + q * 2, (unsigned long long)sh);
            atomicAdd(gp.vacc + (size_t)ord * 6 + q * 2 + 1, (unsigned long long)sl);
        }
    }
}
__global__ void __launch_bounds__(kBlock) k_ground_scatter(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    ground_scatter(a, gp, blockIdx.x);
}

// Closed-form smallest eigenpair of a symmetric PSD 3x3 matrix (trigonometric method), same operation order
// as smallest_eigvec_sym3 in the oracle.
__device__ __forceinline__ void smallest_eig_sym3(const double a[6], double& lmin, double n[3], double& tr) {
    const double xx = a[0], xy = a[1], xz = a[2], yy = a[3], yz = a[4], zz = a[5];
    tr = xx + yy + zz;
    const double p1 = xy * xy + xz * xz + yz * yz;
    const double q = tr / 3.0;
    const double p2 = (xx - q) * (xx - q) + (yy - q) * (yy - q) + (zz - q) * (zz - q) + 2.0 * p1;
    const double p = sqrt(p2 / 6.0);
    if (!(p > 1e-300)) { lmin = q; n[0] = 0; n[1] = 0; n[2] = 1; return; }
    const double b00 = (xx - q) / p, b11 = (yy - q) / p, b22 = (zz - q) / p, b01 = xy / p, b02 = xz / p, b12 = yz / p;
    double r = (b00 * (b11 * b22 - b12 * b12) - b01 * (b01 * b22 - b12 * b02) + b02 * (b01 * b12 - b11 * b02)) / 2.0;
    r = fmin(1.0, fmax(-1.0, r));
    const double phi = acos(r) / 3.0;
    lmin = q + 2.0 * p * cos(phi + 2.0943951023931954923);
    const double r0[3] = {xx - lmin, xy, xz}, r1[3] = {xy, yy - lmin, yz}, r2[3] = {xz, yz, zz - lmin};
    const double c0[3] = {r0[1] * r1[2] - r0[2] * r1[1], r0[2] * r1[0] - r0[0] * r1[2], r0[0] * r1[1] - r0[1] * r1[0]};
    const double c1[3] = {r0[1] * r2[2] - r0[2] * r2[1], r0[2] * r2[0] - r0[0] * r2[2], r0[0] * r2[1] - r0[1] * r2[0]};
    const double c2[3] = {r1[1] * r2[2] - r1[2] * r2[1], r1[2] * r2[0] - r1[0] * r2[2], r1[0] * r2[1] - r1[1] * r2[0]};
    const double d0 = c0[0] * c0[0] + c0[1] * c0[1] + c0[2] * c0[2], d1 = c1[0] * c1[0] + c1[1] * c1[1] + c1[2] * c1[2], d2 = c2[0] * c2[0] + c2[1] * c2[1] + c2[2] * c2[2];
    const double* c = c0; double d = d0;
    if (d1 > d) { c = c1; d = d1; }
    if (d2 > d) { c = c2; d = d2; }
    if (!(d > 1e-300)) { n[0] = 0; n[1] = 0; n[2] = 1; return; }
    const double inv = 1.0 / sqrt(d);
    n[0] = c[0] * inv; n[1] = c[1] * inv; n[2] = c[2] * inv;
    if (n[2] < 0 || (n[2] == 0 && (n[1] < 0 || (n[1] == 0 && n[0] < 0)))) { n[0] = -n[0]; n[1] = -n[1]; n[2] = -n[2]; }
}

// Visits every raw point within the ball B(q, leaf) (strict, float predicate) through the 27-cell block of
// the ball grid: 9 x-rows, each one contiguous run of the sorted array. One WARP per voxel. Lanes 0..8 fetch the
// bounds of the nine runs at once (one round trip instead of nine dependent ones); the lanes then stride over the
// concatenation of the runs, four independent point loads in flight per lane (balls near the sensor hold thousands
// of points, and a chain of dependent loads is all this loop would otherwise be).
template <typename F>
__device__ __forceinline__ void for_each_in_ball_warp(const FramePtrs& a, const GroundPtrs& gp, const GridDesc& g, float qx, float qy, float qz, int lane, F&& f) {
    int cx = (int)floor(((double)qx - g.ox) * g.inv_h), cy = (int)floor(((double)qy - g.oy) * g.inv_h), cz = (int)floor(((double)qz - g.oz) * g.inv_h);
    cx = min(max(cx, 0), g.nx - 1); cy = min(max(cy, 0), g.ny - 1); cz = min(max(cz, 0), g.nz - 1);
    const int x0 = max(cx - 1, 0), x1 = min(cx + 1, g.nx - 1);
    int rb = 0, len = 0;
    if (lane < 9) {
        const int zz = cz - 1 + lane / 3, yy = cy - 1 + lane % 3;
        if (zz >= 0 && zz < g.nz && yy >= 0 && yy < g.ny) {
            const int base = (zz * g.ny + yy) * g.nx;
            rb = a.cell_start[base + x0];
            len = a.cell_start[base + x1 + 1] - rb;
        }
    }
    int incl = len;  // inclusive prefix of the run lengths over lanes 0..8
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) { const int t = __shfl_up_sync(kFull, incl, o); if (lane >= o) incl += t; }
    const int total = __shfl_sync(kFull, incl, 8);
    // every lane keeps the nine (end position in the concatenation, sorted position minus start in the concatenation)
    int r_end[9], r_delta[9];
#pragma unroll
    for (int k = 0; k < 9; k++) {
        r_end[k] = __shfl_sync(kFull, incl, k);
        r_delta[k] = __shfl_sync(kFull, rb - (incl - len), k);
    }
    auto locate = [&](int j) -> int {  // sorted position of element j of the concatenation
        int d = r_delta[0];
#pragma unroll
        for (int k = 1; k < 9; k++) d = j >= r_end[k - 1] ? r_delta[k] : d;
        return j + d;
    };
    const int last = total - 1;
    for (int j = lane; j < total; j += 128) {
        const int j1 = min(j + 32, last), j2 = min(j + 64, last), j3 = min(j + 96, last);
        const float4 p0 = a.spts[locate(j)], p1 = a.spts[locate(j1)], p2 = a.spts[locate(j2)], p3 = a.spts[locate(j3)];
        if (sqdist3(qx, qy, qz, p0.x, p0.y, p0.z) < gp.r2) f(p0);
        if (j + 32 <= last && sqdist3(qx, qy, qz, p1.x, p1.y, p1.z) < gp.r2) f(p1);
        if (j + 64 <= last && sqdist3(qx, qy, qz, p2.x, p2.y, p2.z) < gp.r2) f(p2);
        if (j + 96 <= last && sqdist3(qx, qy, qz, p3.x, p3.y, p3.z) < gp.r2) f(p3);
    }
}

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// ===================================================================================== G5
// One warp per voxel: centroid, ball statistics (moments of d = p - q in double), acceptance test, bin.
__device__ __forceinline__ void voxel_eval_one(const FramePtrs& a, const GroundPtrs& gp, const GridDesc& g, const int v, const int lane) {
    const double nv = (double)gp.vox_n[v];
    const unsigned long long* acc = gp.vacc + (size_t)v * 6;
    const float qx = (float)join_fixed_mean((long long)acc[0], (long long)acc[1], nv);
    const float qy = (float)join_fixed_mean((long long)acc[2], (long long)acc[3], nv);
    const float qz = (float)join_fixed_mean((long long)acc[4], (long long)acc[5], nv);
    int n = 0;
    double m[3] = {0, 0, 0}, s[6] = {0, 0, 0, 0, 0, 0};
    for_each_in_ball_warp(a, gp, g, qx, qy, qz, lane, [&](const float4& p) {
        const double dx = (double)p.x - (double)qx, dy = (double)p.y - (double)qy, dz = (double)p.z - (double)qz;
        n++;
        m[0] += dx; m[1] += dy; m[2] += dz;
        s[0] += dx * dx; s[1] += dx * dy; s[2] += dx * dz; s[3] += dy * dy; s[4] += dy * dz; s[5] += dz * dz;
    });
    n = __reduce_add_sync(kFull, n);
#pragma unroll
    for (int q = 0; q < 3; q++) m[q] = warp_sum_d(m[q]);
#pragma unroll
    for (int q = 0; q < 6; q++) s[q] = warp_sum_d(s[q]);
    if (lane != 0) return;
    float* info = gp.vox_info + (size_t)v * 8;
    info[0] = qx; info[1] = qy; info[2] = qz;
    float acc_flag = 0.f, keyf = 0.f, n0 = 0.f, n1 = 0.f, n2 = 0.f;
    if (n > 3) {  // cpp:131
        const double nn = (double)n;
        const double S[6] = {s[0] - m[0] * m[0] / nn, s[1] - m[0] * m[1] / nn, s[2] - m[0] * m[2] / nn,
                             s[3] - m[1] * m[1] / nn, s[4] - m[1] * m[2] / nn, s[5] - m[2] * m[2] / nn};
        bool ok;
        long long key;
        if (gp.mode == MOR_GROUND_VOXEL_COV) {
            ok = fabs(S[2]) < 0.001 && fabs(S[4]) < 0.001 && fabs(S[5]) < 0.001;  // cpp:145
            key = (long long)(int)__fmul_rn(qz, 10.0f);                            // cpp:166
            n2 = 1.f;
        } else {
            double lmin, nrm[3], tr;
            smallest_eig_sym3(S, lmin, nrm, tr);
            ok = tr > 0 && (lmin / tr) < (double)gp.planarity && nrm[2] > 0.7;
            n0 = (float)nrm[0]; n1 = (float)nrm[1]; n2 = (float)nrm[2];
            const double off = nrm[0] * (double)qx + nrm[1] * (double)qy + nrm[2] * (double)qz;
            key = (long long)floor(off / (double)gp.bin_width);
        }
        key = min(max(key, -32768ll), 32767ll);
        keyf = (float)key;
        if (ok) { acc_flag = 1.f; atomicAdd(&gp.bin_hist[(int)key + 32768], 1); }
    }
    info[3] = acc_flag; info[4] = keyf; info[5] = n0; info[6] = n1; info[7] = n2;
}
// The number of voxels is only known on the device (and is far below the number of points): a fixed grid of warps
// strides over them instead of launching one warp per point's worth of blocks that would mostly exit.
// Blocks [0, nblocks) of a grid of any size take part.
__device__ __forceinline__ void voxel_eval(const FramePtrs& a, const GroundPtrs& gp, int block, int nblocks) {
    const int lane = threadIdx.x & 31;
    const int nvox = gp.gstate[1], warps = (nblocks * kBlock) >> 5;
    const GridDesc g = *gp.ggrid;
    // (consecutive voxels stay in one block on purpose: their balls overlap, so the block shares them in L1; spreading
    // the dense voxels near the sensor over the SMs instead was measured 30 % slower)
    for (int v = (block * kBlock + threadIdx.x) >> 5; v < nvox; v += warps) voxel_eval_one(a, gp, g, v, lane);
}
__global__ void __launch_bounds__(kBlock) k_voxel_eval(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    voxel_eval(a, gp, blockIdx.x, gridDim.x);
}

// ===================================================================================== G6
// Mode bin (cpp:169-178, tie => smallest key) and the selection threshold; resets the look-back state that the
// clustering stage reuses.
__device__ __forceinline__ void ground_mode(const FramePtrs& a, const GroundPtrs& gp) {
    __shared__ unsigned long long s_best[kSingle / 32];
    const bool ascending = !(gp.mode == MOR_GROUND_VOXEL_COV && gp.bin_gap < 0.f);
    unsigned long long best = 0ull;  // (count << 32) | (65535 - rank-of-key): max => largest count, then smallest key
    for (int t = threadIdx.x; t < 65536; t += kSingle) {
        const int k = ascending ? t : 65535 - t;
        const unsigned cnt = (unsigned)gp.bin_hist[k];
        if (cnt) best = max(best, ((unsigned long long)cnt << 32) | (unsigned)(65535 - t));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(kFull, best, o));
    if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < kSingle / 32; w++) best = max(best, s_best[w]);
        const int cnt = (int)(best >> 32);
        const int t = 65535 - (int)(best & 0xFFFFFFFFull);
        gp.gstate[2] = cnt ? (ascending ? t : 65535 - t) : -1;
        gp.gstate[3] = gp.mode == MOR_GROUND_VOXEL_EIGEN ? max(1, (cnt + 3) / 4) : cnt;
        gp.gstate[0] = 0;
        a.scratch->ticket_ingest = 0; a.scratch->ticket_cells = 0;
    }
    for (int t = threadIdx.x; t < a.tiles_pts; t += kSingle) a.st_ingest[t] = 0ull;
    for (int t = threadIdx.x; t < a.tiles_cells; t += kSingle) a.st_cells[t] = 0ull;
    for (int t = threadIdx.x; t < gp.tiles_vox; t += kSingle) gp.st_vox[t] = 0ull;
    if (threadIdx.x < 3) { a.scratch->box_inv_min[threadIdx.x] = 0u; a.scratch->box_max[threadIdx.x] = 0u; }
}
__global__ void __launch_bounds__(kSingle) k_ground_mode(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    ground_mode(a, gp);
}

// ===================================================================================== G7
// ground = union of the balls of the accepted voxels in the selected bins (cpp:184-191).
__device__ __forceinline__ void ground_mark(const FramePtrs& a, const GroundPtrs& gp, int block, int nblocks) {
    const int lane = threadIdx.x & 31;
    const int nvox = gp.gstate[1], warps = (nblocks * kBlock) >> 5;
    if (gp.gstate[2] < 0) return;
    const GridDesc g = *gp.ggrid;
    for (int v = (block * kBlock + threadIdx.x) >> 5; v < nvox; v += warps) {
        const float* info = gp.vox_info + (size_t)v * 8;
        if (info[3] == 0.f) continue;
        const int k = (int)info[4] + 32768;
        const bool take = gp.mode == MOR_GROUND_VOXEL_EIGEN ? gp.bin_hist[k] >= gp.gstate[3] : k == gp.gstate[2];
        if (!take) continue;
        for_each_in_ball_warp(a, gp, g, info[0], info[1], info[2], lane, [&](const float4& p) { gp.is_ground[__float_as_int(p.w)] = 1; });
    }
}
__global__ void __launch_bounds__(kBlock) k_ground_mark(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    ground_mark(a, gp, blockIdx.x, gridDim.x);
}

// ===================================================================================== G8
// ExtractIndices(negative) (cpp:194-198): stable partition of raw_cloud into cloud / gp_indices. The frame kernel
// takes over from here (phase_bin_cloud).
__device__ __forceinline__ void ground_partition(const FramePtrs& a, const GroundPtrs& gp) {
    __shared__ int s_tile;
    if (threadIdx.x == 0) s_tile = atomicAdd(&a.scratch->ticket_ingest, 1);
    __syncthreads();
    const int tile = s_tile;
    const int nraw = a.counts[MOR_CNT_NT];
    const int last_tile = nraw ? (nraw - 1) / kBlock : 0;
    if (tile > last_tile) return;
    const int r = tile * kBlock + threadIdx.x;
    int cls = 0;
    float4 p = make_float4(0, 0, 0, 0);
    int src = 0;
    if (r < nraw) {
        p = gp.rpts[r];
        src = gp.rsrc[r];
        cls = gp.is_ground[r] ? 2 : 1;
        a.point_class[src] = (uint8_t)cls;
    }
    unsigned long long packed = (cls == 1 ? 1ull : 0ull) | (cls == 2 ? (1ull << 31) : 0ull);
    unsigned long long total;
    const unsigned long long in_block = block_exclusive_scan<unsigned long long>(packed, &total);
    const unsigned long long before = tile_exclusive_prefix(a.st_ingest, tile, total);
    const unsigned long long mine = before + in_block;
    if (cls == 1) {
        const int c = (int)(mine & 0x7FFFFFFFull);
        a.pts[c] = p;
        a.cloud_src[c] = src;
    } else if (cls == 2) {
        const int gi = (int)((mine >> 31) & 0x7FFFFFFFull);
        a.gpts[gi] = p;
        a.gsrc[gi] = src;
    }
    if (tile == last_tile && threadIdx.x == 0) {
        const unsigned long long all = before + total;
        a.counts[MOR_CNT_NC] = (int)(all & 0x7FFFFFFFull);
        a.counts[MOR_CNT_NG] = (int)((all >> 31) & 0x7FFFFFFFull);
    }
}
__global__ void __launch_bounds__(kBlock) k_ground_partition(FramePtrs a, GroundPtrs gp) {
    pdl_prologue();
    ground_partition(a, gp);
}

// ===================================================================================== batched forms
// The same nine stages for S sequences per launch (mor_batch_step_device): blockIdx.y is the sequence, whose arguments
// come from the device arrays P / GP. The point-indexed stages are sized for the largest frame of the batch; in the two
// ticket stages the blocks beyond a sequence's own tile count leave before they draw a ticket, so every sequence sees
// exactly the tickets, look-back tiles and zeroing stride of its single-handle launch. The strided stages accept any
// x-size.
__device__ __forceinline__ unsigned ground_blocks_for(uint32_t n) { return n ? (n + kBlock - 1) / kBlock : 1; }

__global__ void __launch_bounds__(kBlock) k_ingest_raw_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    const FramePtrs& a = P[blockIdx.y];
    const unsigned nb = ground_blocks_for(a.n);
    if (blockIdx.x >= nb) return;
    ingest_raw(a, GP[blockIdx.y], nb);
}
__global__ void __launch_bounds__(kBlock) k_ground_keys_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    ground_keys(P[blockIdx.y], GP[blockIdx.y], blockIdx.x);
}
__global__ void __launch_bounds__(kBlock) k_scan_cells_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    scan_cells(P[blockIdx.y], GP[blockIdx.y].ggrid->ncells);  // over the ball-query grid (k_scan_cells: a.dgrid = gp.ggrid)
}
__global__ void __launch_bounds__(kBlock) k_scan_voxels_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    scan_voxels(P[blockIdx.y], GP[blockIdx.y]);
}
__global__ void __launch_bounds__(kBlock) k_ground_scatter_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    ground_scatter(P[blockIdx.y], GP[blockIdx.y], blockIdx.x);
}
__global__ void __launch_bounds__(kBlock) k_voxel_eval_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    voxel_eval(P[blockIdx.y], GP[blockIdx.y], blockIdx.x, gridDim.x);
}
__global__ void __launch_bounds__(kSingle) k_ground_mode_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    ground_mode(P[blockIdx.y], GP[blockIdx.y]);
}
__global__ void __launch_bounds__(kBlock) k_ground_mark_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    ground_mark(P[blockIdx.y], GP[blockIdx.y], blockIdx.x, gridDim.x);
}
__global__ void __launch_bounds__(kBlock) k_ground_partition_batch(const FramePtrs* __restrict__ P, const GroundPtrs* __restrict__ GP) {
    pdl_prologue();
    const FramePtrs& a = P[blockIdx.y];
    if (blockIdx.x >= ground_blocks_for(a.n)) return;
    ground_partition(a, GP[blockIdx.y]);
}

}  // namespace mor
