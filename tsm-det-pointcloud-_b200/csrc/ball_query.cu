// ball_query.cu -- radius / annulus neighbour query for sm_100a: the entry points and the brute-force search.
//
// Replaces (same idx / idx_cnt, bit for bit):
//   ball_query_kernel_fast          /root/reference/pcdet/ops/pointnet2/pointnet2_batch/src/ball_query_gpu.cu:75-112
//   ball_query_dilated_kernel_fast  ball_query_gpu.cu:138-176
//
// Reference semantics kept: hits are the FIRST `nsample` points in index order with
// d2 < r^2 (dilated: rin^2 <= d2 < rout^2), idx_cnt = min(hits, nsample), the row is
// padded cyclically with its own prefix, and a row without hits is all zeros.
//
// Design: clouds of a useful size are answered through a uniform grid (ball_query_grid.cu).  The brute-force search
// below serves the rest -- clouds under 512 points, clouds whose grid is unusable, and TSMDET_BQ_ALGO=brute -- for the
// batch query and for the stacked (ragged) one of stack_ball_query.cu: one warp per centre, lanes test 32 consecutive
// points per step and append the hits in index order (ballot + popc).  Its kernels differ only in how a centre finds
// its cloud and in the write-back; a cloud the grid answered (header word 9 set) is skipped.
#include <string.h>

#include "common.cuh"
#include "grid.cuh"

int tsm_ball_query_grid(bool dilated, int b, int n, int m, float rin, float rout, int nsample, const float* new_xyz,
                        const float* xyz, int* idx_cnt, int* idx, cudaStream_t stream, const int** grid_hdr);

namespace tsm {

constexpr int BQ_WARPS = 8;

// The first `nsample` hits, in index order, of the centre (cx, cy, cz) among the n points (N,3) of one cloud, written to
// row[0..cnt) as index + off; returns cnt = min(hits, nsample) and the first hit's index in `first` (0 without hits).
template <bool DILATED>
__device__ __forceinline__ int brute_query_core(int lane, int n, const float* __restrict__ pts, float cx, float cy,
                                                float cz, float rin2, float rout2, int nsample, int* const row, int off,
                                                int& first) {
    int cnt = 0;
    first = 0;
    for (int base = 0; base < n && cnt < nsample; base += 32) {
        const int k = base + lane;
        bool hit = false;
        if (k < n) {
            const float d2 = sqdist3(__ldg(pts + 3 * k), __ldg(pts + 3 * k + 1), __ldg(pts + 3 * k + 2), cx, cy, cz);
            hit = DILATED ? (d2 >= rin2 && d2 < rout2) : (d2 < rout2);
        }
        const unsigned bal = __ballot_sync(FULL, hit);
        if (bal) {
            if (cnt == 0) first = base + __ffs(bal) - 1;
            const int pos = cnt + __popc(bal & ((1u << lane) - 1u));
            if (hit && pos < nsample) row[pos] = k + off;
            cnt += __popc(bal);
        }
    }
    return min(cnt, nsample);
}

// Batch clouds (b, n, 3): CTA (x, cloud) holds BQ_WARPS warps that stride over the cloud's centres.
template <bool DILATED>
__global__ void __launch_bounds__(BQ_WARPS * 32)
    ball_query_brute_kernel(int n, int m, float rin2, float rout2, int nsample, const float* __restrict__ new_xyz,
                            const float* __restrict__ xyz, const int* __restrict__ grid_hdr, int* __restrict__ idx_cnt,
                            int* __restrict__ idx) {
    const int lane = threadIdx.x & 31;
    const int cloud = blockIdx.y;
    if (grid_hdr && grid_hdr[cloud * kHdrInts + 9]) return;  // answered by the grid query
    const float* const pts = xyz + (size_t)cloud * n * 3;
    for (int c = blockIdx.x * BQ_WARPS + (threadIdx.x >> 5); c < m; c += gridDim.x * BQ_WARPS) {
        const size_t wid = (size_t)cloud * m + c;
        const float cx = __ldg(new_xyz + wid * 3), cy = __ldg(new_xyz + wid * 3 + 1), cz = __ldg(new_xyz + wid * 3 + 2);
        int* const row = idx + wid * nsample;
        int first;
        const int cnt = brute_query_core<DILATED>(lane, n, pts, cx, cy, cz, rin2, rout2, nsample, row, 0, first);
        // count + cyclic padding (row[p] = row[p mod cnt]); a row without hits is zeroed
        __syncwarp();  // the prefix was written by whichever lanes owned it
        if (lane == 0) idx_cnt[wid] = cnt;
        if (cnt == 0) {
            for (int p = lane; p < nsample; p += 32) row[p] = 0;
        } else if (cnt < nsample) {
            for (int p = cnt + lane; p < nsample; p += 32) row[p] = row[p % cnt];
        }
    }
}

// Stacked (ragged) frames, one warp per centre, ball_query_kernel_stack's contract (bq_grid_query16_ragged_kernel in
// ball_query_grid.cu spells it out): frame-local hits padded with the first one, only row[0] = -1 for an empty ball;
// global_rows != 0: frame start + index, all-zero rows for empty balls.  idx_cnt may be null.
__global__ void __launch_bounds__(BQ_WARPS * 32)
    stack_ball_query_kernel(int b, int m, float r2, int nsample, const float* __restrict__ new_xyz,
                            const int* __restrict__ mstart, const int* __restrict__ nstart,
                            const float* __restrict__ xyz, const int* __restrict__ grid_hdr, int* __restrict__ idx_cnt,
                            int* __restrict__ idx, int global_rows) {
    const int lane = threadIdx.x & 31;
    const int centre = blockIdx.x * BQ_WARPS + (threadIdx.x >> 5);
    if (centre >= m) return;
    const int f = stack_frame_of(centre, b, mstart);
    if (grid_hdr && grid_hdr[f * kHdrInts + 9]) return;  // answered by the grid query
    const int start = __ldg(nstart + f), n = __ldg(nstart + f + 1) - start;
    const float cx = __ldg(new_xyz + (size_t)centre * 3), cy = __ldg(new_xyz + (size_t)centre * 3 + 1),
                cz = __ldg(new_xyz + (size_t)centre * 3 + 2);
    int* const row = idx + (size_t)centre * nsample;
    const int off = global_rows ? start : 0;
    int first;
    const int cnt = brute_query_core<false>(lane, n, xyz + (size_t)start * 3, cx, cy, cz, 0.f, r2, nsample, row, off,
                                            first);
    if (idx_cnt && lane == 0) idx_cnt[centre] = cnt;
    if (cnt == 0) {
        if (global_rows)
            for (int p = lane; p < nsample; p += 32) row[p] = 0;
        else if (lane == 0)
            row[0] = -1;
    } else {
        for (int p = cnt + lane; p < nsample; p += 32) row[p] = first + off;
    }
}

}  // namespace tsm

int tsm_stack_ball_query_brute(int b, int m, float radius, int nsample, const float* new_xyz, const int* mstart,
                               const int* nstart, const float* xyz, const int* grid_hdr, int* idx, int* idx_cnt,
                               int global_rows, cudaStream_t stream) {
    using namespace tsm;
    stack_ball_query_kernel<<<(unsigned)divup(m, BQ_WARPS), BQ_WARPS * 32, 0, stream>>>(
        b, m, radius * radius, nsample, new_xyz, mstart, nstart, xyz, grid_hdr, idx_cnt, idx, global_rows);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

static int run_ball_query(bool dilated, int b, int n, int m, float rin, float rout, int nsample, const float* new_xyz,
                          const float* xyz, int* idx_cnt, int* idx, cudaStream_t stream) {
    using namespace tsm;
    if (b <= 0 || m <= 0) return TSM_OK;
    if (n < 0 || nsample <= 0 || b > 65535) return TSM_ERR_INVALID;
    const float rin2 = rin * rin;    // f32 products, as ball_query_gpu.cu:91, 154-155
    const float rout2 = rout * rout;
    // The grid query answers every cloud whose grid is usable and flags it on the device; the brute-force kernel then
    // exits at once for those clouds (no host synchronisation either way).  TSMDET_BQ_ALGO=brute disables the grid.
    const int* ghdr = nullptr;
    const char* algo = tsm_knob(KNOB_BQ_ALGO);
    if (n >= 512 && !(algo && !strcmp(algo, "brute"))) {
        const int rc = tsm_ball_query_grid(dilated, b, n, m, rin, rout, nsample, new_xyz, xyz, idx_cnt, idx, stream,
                                           &ghdr);
        if (rc != TSM_OK) return rc;
    }
    // 16 centres per warp: a CTA for every 128 centres keeps the launch small where the grid answered every cloud
    const dim3 grid((unsigned)divup(m, BQ_WARPS * 16), (unsigned)b);
    if (dilated)
        ball_query_brute_kernel<true><<<grid, BQ_WARPS * 32, 0, stream>>>(n, m, rin2, rout2, nsample, new_xyz, xyz, ghdr,
                                                                          idx_cnt, idx);
    else
        ball_query_brute_kernel<false><<<grid, BQ_WARPS * 32, 0, stream>>>(n, m, rin2, rout2, nsample, new_xyz, xyz, ghdr,
                                                                           idx_cnt, idx);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

extern "C" {

int tsmdet_ball_query(int b, int n, int m, float radius, int nsample, const float* new_xyz, const float* xyz,
                      int* idx_cnt, int* idx, void* stream) {
    return run_ball_query(false, b, n, m, 0.f, radius, nsample, new_xyz, xyz, idx_cnt, idx, (cudaStream_t)stream);
}

int tsmdet_ball_query_dilated(int b, int n, int m, float radius_in, float radius_out, int nsample,
                              const float* new_xyz, const float* xyz, int* idx_cnt, int* idx, void* stream) {
    return run_ball_query(true, b, n, m, radius_in, radius_out, nsample, new_xyz, xyz, idx_cnt, idx,
                          (cudaStream_t)stream);
}

}  // extern "C"
