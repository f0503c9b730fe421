// three_nn_grid.cu -- the three nearest known points of every unknown point, through a uniform grid (sm_100a).
//
// Same dist2 / idx, bit for bit, as three_nn_kernel_fast
//   /root/reference/pcdet/ops/pointnet2/pointnet2_batch/src/interpolate_gpu.cu:16-59
// (strict-< cascade over ascending k: the result is the three lexicographically smallest (d2, k) pairs), without
// its n*m distance tests.  The known points are binned by bq_grid_build_kernel (cells sized for about two points
// each, every cell in ascending index order); one thread per unknown point scans the 3x3x3 cube of cells around
// it and then shell after shell, inserting candidates by (d2, k), until its third-best distance is strictly
// below the distance to the nearest face of the scanned cube that still has cells behind it (with a 2e-4
// relative safety margin on that bound, far above the rounding of the cell coordinates) -- nothing outside the
// cube can then enter the result, ties included.  Clouds whose grid is unusable are left to the brute-force
// kernel (interpolate.cu), which skips the others.
//
// Stacked (ragged) frames, pointnet2_stack's three_nn: one grid per frame over its own known points
// (tsm_grid_build_ragged, the build the stacked ball query uses) and three_nn_grid_ragged_kernel runs the same search
// (three_nn_grid_core); it differs only in finding the unknown point's frame and in adding the frame's known start to
// the indices.  Unusable frames go to stack_three_nn_kernel (stack_interpolate.cu).
#include "grid.cuh"

namespace tsm {

// The three smallest (d2, k) pairs of the unknown point (ux, uy, uz) in one cloud's grid (cell starts cs, index-sorted
// records `sorted` whose w holds the cloud-local index): (b1, i1) <= (b2, i2) <= (b3, i3), +inf / 0 past the cloud's
// points.  The cloud's arrays come as base + offset, not as offset pointers: so three_nn_grid_kernel compiles to the same
// SASS as before the core was factored out of it.
__device__ __forceinline__ void three_nn_grid_core(const GridHdr& h, const int* cell_start_all, size_t cs_off,
                                                   const float4* sorted_all, size_t s_off, float ux, float uy, float uz,
                                                   float& b1, float& b2, float& b3, int& i1, int& i2, int& i3) {
    const int* __restrict__ cs = cell_start_all + cs_off;
    const float4* __restrict__ sorted = sorted_all + s_off;
    // cell coordinates (clamped) and the scaled position used for the face distances
    const float fx = __fmul_rn(__fsub_rn(ux, h.lo[0]), h.inv[0]);
    const float fy = __fmul_rn(__fsub_rn(uy, h.lo[1]), h.inv[1]);
    const float fz = __fmul_rn(__fsub_rn(uz, h.lo[2]), h.inv[2]);
    const int cx = grid_q(ux, h.lo[0], h.inv[0], h.n[0]);
    const int cy = grid_q(uy, h.lo[1], h.inv[1], h.n[1]);
    const int cz = grid_q(uz, h.lo[2], h.inv[2], h.n[2]);
    const float inf = __int_as_float(0x7f800000);
    b1 = inf; b2 = inf; b3 = inf;  // (float)1e40 == +inf: what the reference's double 1e40 becomes in dist2
    i1 = 0; i2 = 0; i3 = 0;

    auto scan = [&](int s0, int s1) {
        for (int p = s0; p < s1; ++p) {
            const float4 v = sorted[p];
            const float d = sqdist3(v.x, v.y, v.z, ux, uy, uz);
            const int k = __float_as_int(v.w);
            if (d < b3 || (d == b3 && k < i3)) {
                if (d < b1 || (d == b1 && k < i1)) {
                    b3 = b2; i3 = i2;
                    b2 = b1; i2 = i1;
                    b1 = d; i1 = k;
                } else if (d < b2 || (d == b2 && k < i2)) {
                    b3 = b2; i3 = i2;
                    b2 = d; i2 = k;
                } else {
                    b3 = d; i3 = k;
                }
            }
        }
    };

    const int rmax = max(max(h.n[0], h.n[1]), h.n[2]);
    for (int R = 1; R <= rmax; ++R) {
        const int z0 = max(cz - R, 0), z1 = min(cz + R, h.n[2] - 1);
        const int y0 = max(cy - R, 0), y1 = min(cy + R, h.n[1] - 1);
        const int x0 = max(cx - R, 0), x1 = min(cx + R, h.n[0] - 1);
        for (int z = z0; z <= z1; ++z) {
            const bool zshell = (z == cz - R) || (z == cz + R);
            for (int y = y0; y <= y1; ++y) {
                const int row = (z * h.n[1] + y) * h.n[0];
                if (R == 1 || zshell || y == cy - R || y == cy + R) {
                    scan(__ldg(cs + row + x0), __ldg(cs + row + x1 + 1));  // the whole x run is new (or R == 1)
                } else {  // interior row of the shell: only its two end cells are new
                    if (cx - R >= 0) scan(__ldg(cs + row + cx - R), __ldg(cs + row + cx - R + 1));
                    if (cx + R < h.n[0]) scan(__ldg(cs + row + cx + R), __ldg(cs + row + cx + R + 1));
                }
            }
        }
        // nearest face of the scanned cube that still has cells behind it; kSlack (in cells) covers the rounding of
        // the scaled coordinates (<= 2048 cells per axis: absolute error below 1e-3 of a cell)
        constexpr float kSlack = 2e-3f;
        float lb = inf;
        if (cx - R > 0) lb = fminf(lb, (fx - (float)(cx - R) - kSlack) / h.inv[0]);
        if (cx + R + 1 < h.n[0]) lb = fminf(lb, ((float)(cx + R + 1) - fx - kSlack) / h.inv[0]);
        if (cy - R > 0) lb = fminf(lb, (fy - (float)(cy - R) - kSlack) / h.inv[1]);
        if (cy + R + 1 < h.n[1]) lb = fminf(lb, ((float)(cy + R + 1) - fy - kSlack) / h.inv[1]);
        if (cz - R > 0) lb = fminf(lb, (fz - (float)(cz - R) - kSlack) / h.inv[2]);
        if (cz + R + 1 < h.n[2]) lb = fminf(lb, ((float)(cz + R + 1) - fz - kSlack) / h.inv[2]);
        if (lb == inf) break;  // the cube covers the grid
        if (lb > 0.f) {
            const float safe = lb * (1.f - 2e-4f);
            if (b3 < safe * safe) break;  // strictly closer than anything outside the cube: ties cannot come from there
        }
    }
}

__global__ void __launch_bounds__(256)
    three_nn_grid_kernel(int n, int m, const float* __restrict__ unknown, const int* __restrict__ hdr_all,
                         const int* __restrict__ cell_start_all, const float4* __restrict__ sorted_all,
                         float* __restrict__ dist2, int* __restrict__ idx) {
    const int b = blockIdx.y;
    const GridHdr h = *reinterpret_cast<const GridHdr*>(hdr_all + (size_t)b * kHdrInts);
    if (!h.ok) return;
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const float* q = unknown + ((size_t)b * n + i) * 3;
    const float ux = __ldg(q), uy = __ldg(q + 1), uz = __ldg(q + 2);
    float b1, b2, b3;
    int i1, i2, i3;
    three_nn_grid_core(h, cell_start_all, (size_t)b * (kGridCells + 1), sorted_all, (size_t)b * m, ux, uy, uz, b1, b2, b3,
                       i1, i2, i3);
    float* od = dist2 + ((size_t)b * n + i) * 3;
    int* oi = idx + ((size_t)b * n + i) * 3;
    od[0] = b1; od[1] = b2; od[2] = b3;
    oi[0] = i1; oi[1] = i2; oi[2] = i3;
}

// Stacked (ragged) frames, pointnet2_stack's three_nn_kernel_stack contract: unknown row p belongs to frame
// stack_frame_of(p) (ustart = the exclusive prefix sums of the unknown counts) and is answered from that frame's known
// points; idx holds GLOBAL known rows (frame-local index + kstart[f]).  Frames whose grid is unusable are left to
// stack_three_nn_kernel (stack_interpolate.cu).
__global__ void __launch_bounds__(256)
    three_nn_grid_ragged_kernel(int b, int n, const float* __restrict__ unknown, const int* __restrict__ ustart,
                                const int* __restrict__ kstart, const int* __restrict__ hdr_all,
                                const int* __restrict__ cell_start_all, const float4* __restrict__ sorted_all,
                                float* __restrict__ dist2, int* __restrict__ idx) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= n) return;
    const int f = stack_frame_of(i, b, ustart);
    const GridHdr h = *reinterpret_cast<const GridHdr*>(hdr_all + (size_t)f * kHdrInts);
    if (!h.ok) return;
    const int start = __ldg(kstart + f);
    const float* q = unknown + (size_t)i * 3;
    const float ux = __ldg(q), uy = __ldg(q + 1), uz = __ldg(q + 2);
    float b1, b2, b3;
    int i1, i2, i3;
    three_nn_grid_core(h, cell_start_all, (size_t)f * (kGridCells + 1), sorted_all, (size_t)start, ux, uy, uz, b1, b2, b3,
                       i1, i2, i3);
    float* od = dist2 + (size_t)i * 3;
    int* oi = idx + (size_t)i * 3;
    od[0] = b1; od[1] = b2; od[2] = b3;
    oi[0] = i1 + start; oi[1] = i2 + start; oi[2] = i3 + start;
}

}  // namespace tsm

// Answers every cloud whose grid is usable; *grid_hdr is what the brute-force kernel consults to skip them.
int tsm_three_nn_grid(int b, int n, int m, const float* unknown, const float* known, float* dist2, int* idx,
                      cudaStream_t stream, const int** grid_hdr) {
    using namespace tsm;
    const int *hdr = nullptr, *cell_start = nullptr;
    const float4* sorted = nullptr;
    int rc = tsm_grid_build(b, m, -1.f, known, stream, 5, &hdr, &cell_start, &sorted);
    if (rc != TSM_OK) return rc;
    dim3 grid((unsigned)divup(n, 256), (unsigned)b);
    three_nn_grid_kernel<<<grid, 256, 0, stream>>>(n, m, unknown, hdr, cell_start, sorted, dist2, idx);
    TSM_LAUNCH_CHECK();
    *grid_hdr = hdr;
    return TSM_OK;
}

// Stacked frames (grid.cuh); the grids use scratch tag 11, apart from the stacked ball query's 9.
int tsm_stack_three_nn_grid(int b, int n, int m, const float* unknown, const int* ustart, const float* known,
                            const int* kstart, float* dist2, int* idx, cudaStream_t stream, const int** grid_hdr) {
    using namespace tsm;
    const int *hdr = nullptr, *cell_start = nullptr;
    const float4* sorted = nullptr;
    int rc = tsm_grid_build_ragged(b, m, -1.f, kstart, known, stream, 11, &hdr, &cell_start, &sorted);
    if (rc != TSM_OK) return rc;
    three_nn_grid_ragged_kernel<<<(unsigned)divup(n, 256), 256, 0, stream>>>(b, n, unknown, ustart, kstart, hdr, cell_start,
                                                                           sorted, dist2, idx);
    TSM_LAUNCH_CHECK();
    *grid_hdr = hdr;
    return TSM_OK;
}
