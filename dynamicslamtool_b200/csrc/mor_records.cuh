// mor_records.cuh — the filtered cloud in the input's own record layout (mor_set_output_records).
//
// A stand-alone gather after the frame kernel: it replays the filter phase's stable compaction over the items
// [cloud | ground] (cpp:673-684) and copies, for every kept item, the point_step bytes of the input record the item came
// from. Output positions therefore equal those of the pcl::PointXYZI records the filter phase wrote. The frame kernels are
// not touched, so the default output path is the same code as without this file.
//
// keep(t) is the filter phase's own predicate: a `cloud` item survives unless ExtractIndices overflowed or its cluster was
// selected (cluster_removed, written by the filter phase's writer CTA); a ground item always survives. (The removal mask
// is not used: a repeated filterCloud only ever sets entries of it, so after a repeat it can still mark points of a cluster
// that is no longer selected.)
#pragma once
#include "mor_kernels.cuh"

namespace mor {

constexpr int kRecT = 1024;     // threads per block = items per tile
enum RecCopy { REC_VEC16 = 0, REC_WORD = 1, REC_BYTES = 2 };

struct RecordPtrs {
    const uint8_t* in; uint32_t step; int copy;  // RecCopy: what the alignment of in / out / step allows
    const int* counts; const int* cid; const uint8_t* cluster_removed; const TrackState* track;
    const int* cloud_src; const int* gsrc;       // item -> input index (frame-parity buffers of the back half)
    uint8_t* out;
    unsigned long long* st;  // [blocks of the launch] look-back tile states, all zero between launches
    int* ctr;                // [0] tile ticket, [1] blocks done: zero between launches
};

// Byte d of the tile's destination range: byte d % step of the record of its (d / step)-th kept item.
__device__ __forceinline__ uint8_t rec_byte(const RecordPtrs& r, const int* src, uint32_t d) {
    const uint32_t k = d / r.step;
    return r.in[(size_t)src[k] * r.step + (d - k * r.step)];
}

// The tile's kept records land in one contiguous byte range [lo, lo + len) of the output. Coalesced aligned stores; in
// the bytewise mode the words at both ends of the range are shared with the neighbouring tiles and are written byte by
// byte, so no two blocks store to one word.
__device__ __forceinline__ void copy_records(const RecordPtrs& r, const int* src, size_t lo, int cnt) {
    const uint32_t step = r.step, len = (uint32_t)cnt * step;
    uint8_t* dst = r.out + lo;
    if (r.copy == REC_VEC16) {
        for (uint32_t d = threadIdx.x * 16u; d < len; d += kRecT * 16u) {
            const uint32_t k = d / step;
            *reinterpret_cast<uint4*>(dst + d) = *reinterpret_cast<const uint4*>(r.in + (size_t)src[k] * step + (d - k * step));
        }
        return;
    }
    if (r.copy == REC_WORD) {
        for (uint32_t d = threadIdx.x * 4u; d < len; d += kRecT * 4u) {
            const uint32_t k = d / step;
            *reinterpret_cast<uint32_t*>(dst + d) = *reinterpret_cast<const uint32_t*>(r.in + (size_t)src[k] * step + (d - k * step));
        }
        return;
    }
    const uint32_t head = (uint32_t)((4u - ((uintptr_t)dst & 3u)) & 3u);
    if (head >= len) {
        for (uint32_t d = threadIdx.x; d < len; d += kRecT) dst[d] = rec_byte(r, src, d);
        return;
    }
    const uint32_t words = (len - head) / 4u, tail = head + words * 4u;
    if (threadIdx.x < head) dst[threadIdx.x] = rec_byte(r, src, threadIdx.x);
    if (tail + threadIdx.x < len) dst[tail + threadIdx.x] = rec_byte(r, src, tail + threadIdx.x);
    for (uint32_t w = threadIdx.x; w < words; w += kRecT) {
        uint32_t d = head + w * 4u, k = d / step, o = d - k * step, v = 0;
#pragma unroll
        for (int b = 0; b < 4; b++) {
            if (o == step) { k++; o = 0; }
            v |= (uint32_t)r.in[(size_t)src[k] * step + o] << (8 * b);
            o++;
        }
        *reinterpret_cast<uint32_t*>(dst + d) = v;
    }
}

// One tile per block, tiles by ticket (every tile a block waits for belongs to a block that is already running); the
// last block out puts the tile states and counters back to zero.
__device__ __forceinline__ void gather_records(const RecordPtrs& r) {
    __shared__ int s_src[kRecT];
    __shared__ int s_tile, s_last;
    if (threadIdx.x == 0) s_tile = atomicAdd(&r.ctr[0], 1);
    __syncthreads();
    const int tile = s_tile;
    const int nc = r.counts[MOR_CNT_NC], total = nc + r.counts[MOR_CNT_NG];
    const int last_tile = total ? (total - 1) / kRecT : 0;
    if (tile <= last_tile) {
        const int t = tile * kRecT + (int)threadIdx.x;
        bool keep = false;
        int src = 0;
        if (t < nc) {
            const int c = r.cid[t];
            keep = !(r.track->extract_overflow || (c >= 0 && r.cluster_removed[c]));
            src = r.cloud_src[t];
        } else if (t < total) {
            keep = true;
            src = r.gsrc[t - nc];
        }
        int cnt;
        const int in_block = block_exclusive_scan<int, kRecT>(keep ? 1 : 0, &cnt);
        const unsigned long long before = tile_prefix_wide<kRecT>(r.st, tile, (unsigned long long)cnt);
        if (keep) s_src[in_block] = src;
        __syncthreads();
        copy_records(r, s_src, (size_t)before * r.step, cnt);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = atomicAdd(&r.ctr[1], 1) == (int)gridDim.x - 1;
        __threadfence();
    }
    __syncthreads();
    if (!s_last) return;
    for (int i = threadIdx.x; i < (int)gridDim.x; i += kRecT) r.st[i] = 0ull;
    if (threadIdx.x == 0) { r.ctr[0] = 0; r.ctr[1] = 0; }
}

__global__ void __launch_bounds__(kRecT, 1) k_gather_records(const __grid_constant__ RecordPtrs r) { gather_records(r); }

// mor_batch_step_device: blockIdx.y = sequence; the x-size fits the largest frame of the batch, and every block of a
// sequence draws a ticket of that sequence, so each sequence resets exactly the states it used.
__global__ void __launch_bounds__(kRecT, 1) k_gather_records_batch(const RecordPtrs* __restrict__ R) { gather_records(R[blockIdx.y]); }

}  // namespace mor
