// mor_batch_mixed.cu — the kernels of mor_batch_step_device_mixed: the frame kernel for S sequences in CTA groups of
// uneven size, and the gather of output records for sequences with limits of their own.
//
// They have a translation unit of their own, because a kernel added to mor_b200.cu's module changes the code of kernels
// already there: the LK frame kernel calls the out-of-line large-K steps (phase_select_large, phase_match_large,
// phase_filter_large), and one more caller changes how ptxas compiles them and every LK kernel that calls them. The
// device code is included
// under a namespace of its own, so that none of its symbols (kernel stubs, the host stubs of out-of-line device
// functions) collides with mor_b200.cu's at link time; the arguments cross over as device addresses.
#include <cuda_runtime.h>

#define mor mor_mixed_tu
#include "mor_kernels.cuh"
#include "mor_records.cuh"
#undef mor

namespace mor_mixed_tu {

// T[g] = {first CTA, size G_g, begin, end} for the `groups` groups in ascending first CTA, followed by the sequence order
// (ints): group g steps the sequences order[begin .. end) in turn on its G_g CTAs. Each sequence's edge segments were
// cut for its own group's G_g (set_segments).
template <bool LK>
__global__ void __launch_bounds__(kT, 1) k_frame_batch_mixed(const FramePtrs* __restrict__ P, const int4* __restrict__ T, int groups) {
    extern __shared__ __align__(128) unsigned long long dyn[];
    __shared__ FilterShared sh;
    int lo = 0, hi = groups - 1;  // the last group whose first CTA is at or below this one
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (T[mid].x <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
    }
    const int4 grp = T[lo];
    const int* order = reinterpret_cast<const int*>(T + groups);
    for (int i = grp.z; i < grp.w; i++) frame_body<LK>(P[order[i]], (int)blockIdx.x - grp.x, grp.y, sh, dyn);
}

// gather_records (mor_records.cuh) for a batch whose handles' limits differ: a sequence's tile states are sized for its own
// max_points, so they may be fewer than the launch's x-size, which fits the largest frame. The blocks beyond the
// sequence's own count nb[y] leave before they draw a ticket, and the last of its own blocks out resets exactly those
// states; the rest is gather_records line for line. (A copy rather than a parameter of gather_records: one changes the
// code of k_gather_records and k_gather_records_batch.)
__global__ void __launch_bounds__(kRecT, 1) k_gather_records_mixed(const RecordPtrs* __restrict__ R, const int* __restrict__ nb) {
    const int blocks = nb[blockIdx.y];
    if ((int)blockIdx.x >= blocks) return;
    const RecordPtrs& r = R[blockIdx.y];
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
        s_last = atomicAdd(&r.ctr[1], 1) == blocks - 1;
        __threadfence();
    }
    __syncthreads();
    if (!s_last) return;
    for (int i = threadIdx.x; i < blocks; i += kRecT) r.st[i] = 0ull;
    if (threadIdx.x == 0) { r.ctr[0] = 0; r.ctr[1] = 0; }
}

}  // namespace mor_mixed_tu

namespace mor {

cudaError_t configure_frame_batch_mixed(size_t smem) {
    using namespace mor_mixed_tu;
    cudaError_t e = cudaFuncSetAttribute(k_frame_batch_mixed<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    return e != cudaSuccess ? e : cudaFuncSetAttribute(k_frame_batch_mixed<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
}

cudaError_t launch_frame_batch_mixed(bool lk, unsigned grid, size_t smem, cudaStream_t st, const void* P, const void* T, int groups) {
    using namespace mor_mixed_tu;
    void* argv[] = {(void*)&P, (void*)&T, (void*)&groups};
    const void* kernel = lk ? (const void*)k_frame_batch_mixed<true> : (const void*)k_frame_batch_mixed<false>;
    return cudaLaunchCooperativeKernel(kernel, dim3(grid), dim3(mor_mixed_tu::kT), argv, smem, st);
}

cudaError_t launch_gather_records_mixed(unsigned blocks_x, unsigned seqs, cudaStream_t st, const void* R, const void* nb) {
    using namespace mor_mixed_tu;
    k_gather_records_mixed<<<dim3(blocks_x, seqs), kRecT, 0, st>>>(static_cast<const RecordPtrs*>(R), static_cast<const int*>(nb));
    return cudaGetLastError();
}

}  // namespace mor
