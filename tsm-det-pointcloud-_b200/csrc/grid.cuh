// grid.cuh -- the per-cloud uniform grid shared by the grid ball query and the grid 3-NN (built by
// bq_grid_build_kernel in ball_query_grid.cu).
#pragma once
#include "common.cuh"

namespace tsm {

constexpr int kGridCells = 32768;   // shared-memory histogram: 128 KB
constexpr int kMaxCell = 256;       // largest cell population the index fix-up accepts
constexpr int kHdrInts = 16;        // per-cloud header: lo[3], inv[3] (float bits), n[3], ok

struct GridHdr {
    float lo[3];
    float inv[3];
    int n[3];
    int ok;
};

__device__ __forceinline__ int grid_q(float v, float lo, float inv, int n) {
    return min(max(__float2int_rd(__fmul_rn(__fsub_rn(v, lo), inv)), 0), n - 1);
}

// Frame of row p of a stacked (ragged) batch, as ball_query_kernel_stack finds it: the first k with
// p < M0 + ... + Mk, the search stopping at b - 1.  mstart = the (b + 1) exclusive prefix sums of the counts.
__device__ __forceinline__ int stack_frame_of(int p, int b, const int* __restrict__ mstart) {
    int lo = 0, hi = b - 1;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (p < __ldg(mstart + mid + 1)) hi = mid; else lo = mid + 1;
    }
    return lo;
}

}  // namespace tsm

// Builds the grid of every cloud on `stream` (scratch tag `tag`): cells at least 1.01 * rout wide, or -- rout < 0 --
// sized for about two points per cell.  Returns device pointers into the scratch buffer.
int tsm_grid_build(int b, int n, float rout, const float* xyz, cudaStream_t stream, int tag, const int** hdr,
                   const int** cell_start, const float4** sorted);

// Stacked clouds: one grid per frame over its own points (start = the (b + 1) exclusive prefix sums of the counts, on the
// device; n_total points in all), same cell sizing as tsm_grid_build.  A frame's sorted records begin at sorted + start[f]
// and carry frame-local indices; its cell starts are frame-local too.
int tsm_grid_build_ragged(int b, int n_total, float rout, const int* start, const float* xyz, cudaStream_t stream, int tag,
                          const int** hdr, const int** cell_start, const float4** sorted);

// Writes nstart / mstart (b + 1 each, device) = the exclusive prefix sums of the device count arrays ncnt / mcnt
// (stack_ball_query.cu, one launch).
int tsm_stack_counts_scan(int b, const int* ncnt, const int* mcnt, int* nstart, int* mstart, cudaStream_t stream);

// Stacked clouds: one grid per frame over its own points (nstart / mstart = the (b + 1) exclusive prefix sums of the
// point / centre counts, on the device); answers every centre of a frame whose grid is usable.  *grid_hdr receives the
// per-frame headers (word 9 = usable; nullptr: no grid was built) for the brute-force kernel.
int tsm_stack_ball_query_grid(int b, int m, int n_total, float radius, int nsample, const float* new_xyz,
                              const int* mstart, const int* nstart, const float* xyz, int* idx, int* idx_cnt,
                              int global_rows, cudaStream_t stream, const int** grid_hdr);

// Stacked 3-NN (three_nn_grid.cu): one grid per frame over its known points (kstart / ustart = the (b + 1) exclusive prefix
// sums of the known / unknown counts, on the device; m known points in all); answers every unknown point of a frame whose
// grid is usable, with global known rows.  *grid_hdr receives the per-frame headers (word 9 = usable).
int tsm_stack_three_nn_grid(int b, int n, int m, const float* unknown, const int* ustart, const float* known,
                            const int* kstart, float* dist2, int* idx, cudaStream_t stream, const int** grid_hdr);

// Stacked clouds by brute force (ball_query.cu): every centre of a frame whose header word 9 is not set (all of them when
// grid_hdr is nullptr), same arguments and contract as the grid query.
int tsm_stack_ball_query_brute(int b, int m, float radius, int nsample, const float* new_xyz, const int* mstart,
                               const int* nstart, const float* xyz, const int* grid_hdr, int* idx, int* idx_cnt,
                               int global_rows, cudaStream_t stream);
