// stack_ball_query.cu -- ball query over stacked (ragged) frames, pointnet2_stack's ball_query_wrapper, and the
// feature rows that feed a stacked SA scale to the fused MLP kernels.
//
// Replaces (same idx, bit for bit):
//   ball_query_kernel_stack   /root/reference/pcdet/ops/pointnet2/pointnet2_stack/src/ball_query_gpu.cu:15-62
//
// Reference semantics kept: centre p belongs to the first frame k with p < M0 + ... + Mk (the search stops at B - 1);
// its frame's points are scanned in ascending frame-local index, d2 < radius * radius (fp32 product, strict); the first
// hit fills all nsample slots, every hit then goes to slot cnt++, the scan stops at nsample; a centre without hits gets
// only idx[p, 0] = -1.  Indices are frame-local.
//
// Design: the frame starts come from a device-side scan of the two count arrays (no host synchronisation); every frame
// then gets its own uniform grid over its own points (bq_grid_build_ragged_kernel, the same build as the batch grid
// query, ball_query_grid.cu) and is answered by the half-warp / merge grid queries.  Frames whose grid is unusable
// (> kMaxCell points in one cell, a non-finite extent, no points) and TSMDET_BQ_ALGO=brute go to the brute-force
// search of ball_query.cu (stack_ball_query_kernel), which skips the frames the grid answered.
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "grid.cuh"
#include "umma.cuh"

namespace tsm {

// nstart / mstart (b + 1) = exclusive prefix sums of xyz_batch_cnt / new_xyz_batch_cnt; warp 0 scans the points,
// warp 1 the centres.
__global__ void __launch_bounds__(64) stack_counts_scan_kernel(int b, const int* __restrict__ ncnt,
                                                               const int* __restrict__ mcnt, int* __restrict__ nstart,
                                                               int* __restrict__ mstart) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int* const cnt = w ? mcnt : ncnt;
    int* const out = w ? mstart : nstart;
    int carry = 0;
    for (int base = 0; base < b; base += 32) {
        const int i = base + lane;
        const int v = i < b ? __ldg(cnt + i) : 0;
        int inc = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(FULL, inc, o);
            if (lane >= o) inc += t;
        }
        if (i < b) out[i] = carry + inc - v;
        carry += __shfl_sync(FULL, inc, 31);
    }
    if (lane == 0) out[b] = carry;
}

// Stacked features (N,C) fp32 -> rows (N,Cp) in the fused MLP's operand type, zero padded, rounded exactly as
// transpose2_kernel (mlp_tc2.cu) rounds the (B,C,N) planes: bf16 round-to-nearest-even (Cp = round_up(C, 8)) or the
// fp32 bit pattern of tf32 round-half-away (Cp = round_up(C, 4)).  One 4-byte word per thread; both the reads and the
// writes of a warp are contiguous runs.
template <typename OutT>
__global__ void __launch_bounds__(256) stack_feature_rows_kernel(long long n, int c, int cp, const float* __restrict__ f,
                                                                 OutT* __restrict__ out) {
    constexpr int EPW = 4 / (int)sizeof(OutT);  // elements per word
    const int wpr = cp / EPW;
    const long long words = n * wpr;
    uint32_t* const dst = reinterpret_cast<uint32_t*>(out);
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < words; e += (long long)gridDim.x * 256) {
        const long long p = e / wpr;
        const int ch = (int)(e - p * wpr) * EPW;
        const float* const src = f + p * c;
        if constexpr (sizeof(OutT) == 2) {
            const float v0 = ch < c ? __ldg(src + ch) : 0.f, v1 = ch + 1 < c ? __ldg(src + ch + 1) : 0.f;
            const __nv_bfloat162 h = __halves2bfloat162(__float2bfloat16_rn(v0), __float2bfloat16_rn(v1));
            dst[e] = *reinterpret_cast<const uint32_t*>(&h);
        } else {
            dst[e] = to_tf32(ch < c ? __ldg(src + ch) : 0.f);
        }
    }
}

}  // namespace tsm

int tsm_stack_counts_scan(int b, const int* ncnt, const int* mcnt, int* nstart, int* mstart, cudaStream_t stream) {
    tsm::stack_counts_scan_kernel<<<1, 64, 0, stream>>>(b, ncnt, mcnt, nstart, mstart);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

extern "C" {

int tsmdet_stack_ball_query(int b, int m, int n_total, float radius, int nsample, const float* new_xyz,
                            const int* new_xyz_batch_cnt, const float* xyz, const int* xyz_batch_cnt, int* idx,
                            int* idx_cnt, int global_rows, void* stream_) {
    using namespace tsm;
    if (m <= 0) return TSM_OK;
    if (b <= 0 || n_total < 0 || nsample <= 0 || !new_xyz || !new_xyz_batch_cnt || !xyz_batch_cnt || !idx ||
        (n_total > 0 && !xyz))
        return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    void* p = nullptr;
    int rc = tsm_scratch_get(10, sizeof(int) * 2 * ((size_t)b + 1), stream, &p);
    if (rc != TSM_OK) return rc;
    int* const nstart = static_cast<int*>(p);
    int* const mstart = nstart + b + 1;
    rc = tsm_stack_counts_scan(b, xyz_batch_cnt, new_xyz_batch_cnt, nstart, mstart, stream);
    if (rc != TSM_OK) return rc;
    const int* ghdr = nullptr;
    const char* algo = tsm_knob(KNOB_BQ_ALGO);
    if (!(algo && !strcmp(algo, "brute"))) {
        rc = tsm_stack_ball_query_grid(b, m, n_total, radius, nsample, new_xyz, mstart, nstart, xyz, idx, idx_cnt,
                                       global_rows, stream, &ghdr);
        if (rc != TSM_OK) return rc;
    }
    return tsm_stack_ball_query_brute(b, m, radius, nsample, new_xyz, mstart, nstart, xyz, ghdr, idx, idx_cnt, global_rows,
                                      stream);
}

int tsmdet_stack_feature_rows(int precision, int n, int c, const float* features, void* rows, void* stream) {
    using namespace tsm;
    if (n <= 0 || c <= 0) return TSM_OK;
    if (!features || !rows || (precision != 1 && precision != 2)) return TSM_ERR_INVALID;
    const int q = precision == 1 ? 8 : 4;
    const int cp = (c + q - 1) / q * q;
    const long long words = (long long)n * cp / (precision == 1 ? 2 : 1);
    const unsigned grid = (unsigned)std::min<long long>((words + 255) / 256, (long long)tsm_num_sms() * 16);
    if (precision == 1)
        stack_feature_rows_kernel<__nv_bfloat16><<<grid, 256, 0, (cudaStream_t)stream>>>(n, c, cp, features,
                                                                                        (__nv_bfloat16*)rows);
    else
        stack_feature_rows_kernel<float><<<grid, 256, 0, (cudaStream_t)stream>>>(n, c, cp, features, (float*)rows);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

}  // extern "C"
