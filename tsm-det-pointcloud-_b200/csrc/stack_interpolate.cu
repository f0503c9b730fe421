// stack_interpolate.cu -- three_nn / three_interpolate over stacked (ragged) frames, pointnet2_stack's three_nn_wrapper /
// three_interpolate_wrapper / three_interpolate_grad_wrapper (sm_100a).
//
// Replaces (same dist2 / idx / features, bit for bit):
//   three_nn_kernel_stack                /root/reference/pcdet/ops/pointnet2/pointnet2_stack/src/interpolate_gpu.cu
//   three_interpolate_kernel_stack       (same file)
//   three_interpolate_grad_kernel_stack  (same file)
//
// Reference semantics kept: unknown row p belongs to the first frame k with p < N0 + ... + Nk (the search stops at B - 1);
// that frame's known points are scanned in ascending frame-local index with the strict-< cascade (ties keep the earlier
// index), bests starting at 1e40 (+inf in f32); idx holds GLOBAL known rows, and the slots a frame with fewer than three
// known points cannot fill are (+inf, the frame's known start).  Interpolation: out[p,c] = w0 f[i0,c] + w1 f[i1,c] +
// w2 f[i2,c], compiled as fmaf(w2,f2, fmaf(w0,f0, w1*f1)) like the batch kernel.
//
// Design: the frame starts come from the device-side scan of the stacked ball query (no host synchronisation); every
// frame gets its own grid over its known points and is answered by the batch grid 3-NN's search (three_nn_grid.cu).
// Frames whose grid is unusable (no known points, a non-finite coordinate, > kMaxCell points in one cell) and
// TSMDET_NN_ALGO=brute go to stack_three_nn_kernel below, which skips the frames the grid answered.
//
// One deliberate difference: an interpolation index outside [0, M) reads 0 where the reference reads out of bounds.  It
// occurs: an unknown point of a frame without known points gets idx = that frame's known start, which is M when no
// later frame has known points.  Its weights are 0/0 = NaN in the module, so the output is NaN either way.
#include <string.h>

#include "common.cuh"
#include "grid.cuh"

namespace tsm {

// One thread per unknown point, the known points of its frame in ascending index.
__global__ void __launch_bounds__(256)
    stack_three_nn_kernel(int b, int n, const float* __restrict__ unknown, const int* __restrict__ ustart,
                          const float* __restrict__ known, const int* __restrict__ kstart, const int* __restrict__ grid_hdr,
                          float* __restrict__ dist2, int* __restrict__ idx) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int f = stack_frame_of(i, b, ustart);
    if (grid_hdr && grid_hdr[f * kHdrInts + 9]) return;  // answered by the grid search (three_nn_grid.cu)
    const int start = __ldg(kstart + f), mf = __ldg(kstart + f + 1) - start;
    const float* q = unknown + (size_t)i * 3;
    const float ux = __ldg(q), uy = __ldg(q + 1), uz = __ldg(q + 2);
    const float* kn = known + (size_t)start * 3;
    float b1 = __int_as_float(0x7f800000), b2 = b1, b3 = b1;  // (float)1e40 == +inf
    int i1 = 0, i2 = 0, i3 = 0;
    for (int k = 0; k < mf; ++k) {
        const float d = sqdist3(__ldg(kn + 3 * k), __ldg(kn + 3 * k + 1), __ldg(kn + 3 * k + 2), ux, uy, uz);
        if (d < b3) {
            if (d < b1) {
                b3 = b2; i3 = i2;
                b2 = b1; i2 = i1;
                b1 = d; i1 = k;
            } else if (d < b2) {
                b3 = b2; i3 = i2;
                b2 = d; i2 = k;
            } else {
                b3 = d; i3 = k;
            }
        }
    }
    float* od = dist2 + (size_t)i * 3;
    int* oi = idx + (size_t)i * 3;
    od[0] = b1; od[1] = b2; od[2] = b3;
    oi[0] = i1 + start; oi[1] = i2 + start; oi[2] = i3 + start;
}

constexpr int kIpPts = 32;  // points per CTA of the interpolation kernels (8 warps x 4)

// features (M,C) rows, idx / weight (N,3) -> out (N,C) rows (PLANES = false) or (C,N) planes (PLANES = true, the
// point-wise MLP's src0).  A warp owns four points, its lanes run over 32 consecutive channels at a time, so the three
// feature rows are read in contiguous runs; planes go through a 32 x 32 shared-memory transpose so that their writes are
// contiguous too.  Both layouts evaluate the same expression per element.  HBM-bound.
template <bool PLANES>
__global__ void __launch_bounds__(256)
    stack_three_interpolate_kernel(int n, int c, int m, const float* __restrict__ features, const int* __restrict__ idx,
                                   const float* __restrict__ weight, float* __restrict__ out) {
    __shared__ float tile[32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p0 = blockIdx.x * kIpPts;
    int j[4][3];
    float w[4][3];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int p = p0 + warp + 8 * k;
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            j[k][s] = p < n ? __ldg(idx + (size_t)p * 3 + s) : -1;
            w[k][s] = p < n ? __ldg(weight + (size_t)p * 3 + s) : 0.f;
        }
    }
    for (int c0 = 0; c0 < c; c0 += 32) {
        const int ch = c0 + lane;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = p0 + warp + 8 * k;
            float f[3];
#pragma unroll
            for (int s = 0; s < 3; ++s)
                f[s] = ((unsigned)j[k][s] < (unsigned)m && ch < c) ? __ldg(features + (size_t)j[k][s] * c + ch) : 0.f;
            const float v = __fmaf_rn(w[k][2], f[2], __fmaf_rn(w[k][0], f[0], __fmul_rn(w[k][1], f[1])));
            if (PLANES)
                tile[lane][warp + 8 * k] = v;
            else if (p < n && ch < c)
                out[(size_t)p * c + ch] = v;
        }
        if (PLANES) {
            __syncthreads();
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int cc = c0 + warp + 8 * k, p = p0 + lane;
                if (cc < c && p < n) out[(size_t)cc * n + p] = tile[warp + 8 * k][lane];
            }
            __syncthreads();
        }
    }
}

// grad_out (N,C), idx / weight (N,3) -> grad_features (M,C) += g * w (atomic; zeroed by the caller); same layout as the
// forward rows kernel and the same guard on the index.
__global__ void __launch_bounds__(256)
    stack_three_interpolate_grad_kernel(int n, int c, int m, const float* __restrict__ grad_out,
                                        const int* __restrict__ idx, const float* __restrict__ weight,
                                        float* __restrict__ grad_features) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int p = blockIdx.x * kIpPts + warp + 8 * k;
        if (p >= n) return;
        int j[3];
        float w[3];
#pragma unroll
        for (int s = 0; s < 3; ++s) {
            j[s] = __ldg(idx + (size_t)p * 3 + s);
            w[s] = __ldg(weight + (size_t)p * 3 + s);
        }
        for (int ch = lane; ch < c; ch += 32) {
            const float g = __ldg(grad_out + (size_t)p * c + ch);
#pragma unroll
            for (int s = 0; s < 3; ++s)
                if ((unsigned)j[s] < (unsigned)m) atomicAdd(grad_features + (size_t)j[s] * c + ch, __fmul_rn(g, w[s]));
        }
    }
}

}  // namespace tsm

extern "C" {

int tsmdet_stack_three_nn(int b, int n, int m, const float* unknown, const int* unknown_batch_cnt, const float* known,
                          const int* known_batch_cnt, float* dist2, int* idx, void* stream_) {
    using namespace tsm;
    if (n <= 0) return TSM_OK;
    if (b <= 0 || m < 0 || !unknown || !unknown_batch_cnt || !known_batch_cnt || !dist2 || !idx || (m > 0 && !known))
        return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    void* p = nullptr;
    int rc = tsm_scratch_get(12, sizeof(int) * 2 * ((size_t)b + 1), stream, &p);
    if (rc != TSM_OK) return rc;
    int* const kstart = static_cast<int*>(p);
    int* const ustart = kstart + b + 1;
    rc = tsm_stack_counts_scan(b, known_batch_cnt, unknown_batch_cnt, kstart, ustart, stream);
    if (rc != TSM_OK) return rc;
    const int* ghdr = nullptr;
    const char* algo = tsm_knob(KNOB_NN_ALGO);
    if (m > 0 && !(algo && !strcmp(algo, "brute"))) {
        rc = tsm_stack_three_nn_grid(b, n, m, unknown, ustart, known, kstart, dist2, idx, stream, &ghdr);
        if (rc != TSM_OK) return rc;
    }
    stack_three_nn_kernel<<<(unsigned)divup(n, 256), 256, 0, stream>>>(b, n, unknown, ustart, known, kstart, ghdr, dist2,
                                                                      idx);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_stack_three_interpolate(int n, int c, int m, const float* features, const int* idx, const float* weight,
                                   float* out, int planes, void* stream) {
    using namespace tsm;
    if (n <= 0 || c <= 0) return TSM_OK;
    if (m < 0 || !idx || !weight || !out || (m > 0 && !features)) return TSM_ERR_INVALID;
    const unsigned blocks = (unsigned)divup(n, kIpPts);
    if (planes)
        stack_three_interpolate_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(n, c, m, features, idx, weight, out);
    else
        stack_three_interpolate_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(n, c, m, features, idx, weight, out);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_stack_three_interpolate_grad(int n, int c, int m, const float* grad_out, const int* idx, const float* weight,
                                        float* grad_features, void* stream) {
    using namespace tsm;
    if (n <= 0 || c <= 0) return TSM_OK;
    if (m < 0 || !grad_out || !idx || !weight || (m > 0 && !grad_features)) return TSM_ERR_INVALID;
    stack_three_interpolate_grad_kernel<<<(unsigned)divup(n, kIpPts), 256, 0, (cudaStream_t)stream>>>(
        n, c, m, grad_out, idx, weight, grad_features);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

}  // extern "C"
