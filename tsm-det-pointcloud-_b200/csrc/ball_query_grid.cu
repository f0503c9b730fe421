// ball_query_grid.cu -- radius / annulus neighbour query through a uniform grid (sm_100a).
//
// Same results, bit for bit, as ball_query_kernel_fast / ball_query_dilated_kernel_fast
//   /root/reference/pcdet/ops/pointnet2/pointnet2_batch/src/ball_query_gpu.cu:75-112, 138-176
// (first `nsample` points IN INDEX ORDER with d2 < r^2, cyclic padding, zero rows without hits), but
// without the reference's M*N distance tests: only points in the 27 cells around a centre are tested.
//
//  * bq_grid_build_kernel, one CTA per cloud: bounding box -> a grid whose cells are at least 1.01 r wide on
//    every axis and at most 32768 in number (the histogram lives in shared memory) -> counting sort
//    (histogram, scan, scatter) -> a per-cell fix-up that puts every cell's points in ASCENDING ORIGINAL
//    INDEX (each point counts the members of its cell with a smaller index).  Output: cell_start[] and
//    the points as (x, y, z, index) float4 records in cell order.
//  * bq_grid_query16_kernel (nsample <= 32), half a warp per centre, candidate-parallel: see grid_query16_core.
//  * bq_grid_merge_kernel (larger nsample), one warp per centre: lane l < 27 walks the sorted list of one
//    neighbour cell up to its next hit; the warp repeatedly takes the smallest pending index
//    (redux.sync.min) until `nsample` are out.
//    Both evaluate the reference's own distance expression, so the hit set is identical.
//
// A cloud whose points pile up in one cell (> kMaxCell per cell: degenerate input, or r comparable to the
// whole cloud) is flagged and left to the brute-force search of ball_query.cu, which skips flagged-OK
// clouds -- no host synchronisation either way.
//
// Stacked (ragged) frames, pointnet2_stack's ball query: bq_grid_build_ragged_kernel builds one grid per frame over its
// own points and bq_grid_query16_ragged_kernel / bq_grid_merge_ragged_kernel run the same search cores
// (grid_query16_core, grid_merge_core); they differ only in finding the centre's frame and in the write-back (first-hit
// padding, -1 for an empty ball).  Unusable frames go to stack_ball_query_kernel (ball_query.cu).
#include <math.h>

#include "common.cuh"
#include "grid.cuh"

namespace tsm {

// The grid of ONE cloud of n points, built by a whole 1024-thread CTA (the batch and the ragged build kernels below
// differ only in where a cloud's points and outputs start).
__device__ __forceinline__ void grid_build_cloud(int n, float rout, const float* __restrict__ xyz, int* const hdr,
                                                 int* const cell_start, float4* const tmp, float4* const sorted) {
    extern __shared__ __align__(16) unsigned char dyn[];
    uint32_t* const hist = reinterpret_cast<uint32_t*>(dyn);  // [kGridCells]
    __shared__ float red[6][32];
    __shared__ uint32_t woff[32];
    __shared__ uint32_t wmaxc[32];
    constexpr int T = 1024, NW = 32;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;

    // (1) bounding box
    const float inf = __int_as_float(0x7f800000);
    float lo0 = inf, lo1 = inf, lo2 = inf, hi0 = -inf, hi1 = -inf, hi2 = -inf;
    for (int k = tid; k < n; k += T) {
        const float x = __ldg(xyz + 3 * k), y = __ldg(xyz + 3 * k + 1), z = __ldg(xyz + 3 * k + 2);
        lo0 = fminf(lo0, x); hi0 = fmaxf(hi0, x);
        lo1 = fminf(lo1, y); hi1 = fmaxf(hi1, y);
        lo2 = fminf(lo2, z); hi2 = fmaxf(hi2, z);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        lo0 = fminf(lo0, __shfl_xor_sync(FULL, lo0, o)); hi0 = fmaxf(hi0, __shfl_xor_sync(FULL, hi0, o));
        lo1 = fminf(lo1, __shfl_xor_sync(FULL, lo1, o)); hi1 = fmaxf(hi1, __shfl_xor_sync(FULL, hi1, o));
        lo2 = fminf(lo2, __shfl_xor_sync(FULL, lo2, o)); hi2 = fmaxf(hi2, __shfl_xor_sync(FULL, hi2, o));
    }
    if (lane == 0) {
        red[0][warp] = lo0; red[1][warp] = lo1; red[2][warp] = lo2;
        red[3][warp] = hi0; red[4][warp] = hi1; red[5][warp] = hi2;
    }
    for (int c = tid; c < kGridCells; c += T) hist[c] = 0u;
    __syncthreads();
    for (int w = 0; w < NW; ++w) {
        lo0 = fminf(lo0, red[0][w]); lo1 = fminf(lo1, red[1][w]); lo2 = fminf(lo2, red[2][w]);
        hi0 = fmaxf(hi0, red[3][w]); hi1 = fmaxf(hi1, red[4][w]); hi2 = fmaxf(hi2, red[5][w]);
    }
    // (2) grid: cells >= 1.01 r on every axis (so a hit is never more than one cell away, rounding of the
    // cell coordinate included: its error is below 2048 * 2^-22 of a cell), <= 2048 per axis, <= kGridCells
    // in total -- the axis with the smallest extent is coarsened first
    float ext[3] = {hi0 - lo0, hi1 - lo1, hi2 - lo2};
    const float lo[3] = {lo0, lo1, lo2};
    int nc[3];
    const bool automatic = rout < 0.f;  // no radius (3-NN): about two points per cell
    bool ok = automatic || (rout > 0.f && rout < 1.0e18f);
#pragma unroll
    for (int a = 0; a < 3; ++a)
        if (!(ext[a] >= 0.f) || !(ext[a] < 3.0e38f)) { ok = false; ext[a] = 0.f; }
    float s0 = rout * 1.01f;
    if (automatic) {
        // smallest cell edge whose grid has at most `target` cells (bisection; every thread computes the same)
        const float target = fminf(fmaxf(0.5f * (float)n, 64.f), (float)kGridCells);
        float lo_s = 0.f, hi_s = fmaxf(fmaxf(ext[0], ext[1]), ext[2]);
        if (!(hi_s > 0.f)) hi_s = 1.f;
        for (int it = 0; it < 40; ++it) {
            const float mid = 0.5f * (lo_s + hi_s);
            float cells = 1.f;
#pragma unroll
            for (int a = 0; a < 3; ++a) cells *= fminf(fmaxf(floorf(ext[a] / mid), 1.f), 2048.f);
            if (mid > 0.f && cells <= target) hi_s = mid; else lo_s = mid;
        }
        s0 = hi_s;
    }
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        const float q = ok ? floorf(ext[a] / s0) : 1.f;
        nc[a] = (int)fminf(fmaxf(q, 1.f), 2048.f);
    }
    for (int guard = 0; guard < 64 && (long)nc[0] * nc[1] * nc[2] > kGridCells; ++guard) {
        int a = -1;  // smallest-extent axis that still has more than one cell
#pragma unroll
        for (int c = 0; c < 3; ++c)
            if (nc[c] > 1 && (a < 0 || ext[c] < ext[a])) a = c;
        nc[a] = (nc[a] + 1) / 2;
    }
    float inv[3];
#pragma unroll
    for (int a = 0; a < 3; ++a) {
        inv[a] = ext[a] > 0.f ? (float)nc[a] / ext[a] : 0.f;
        // the cell must stay >= 1.01 r after rounding the quotient: shave the scale, never the cell
        if (inv[a] * s0 > 1.f) inv[a] = 1.f / s0;
    }
    const int ncell = nc[0] * nc[1] * nc[2];
    auto cell_of = [&](float x, float y, float z) -> int {
        const int qx = grid_q(x, lo[0], inv[0], nc[0]);
        const int qy = grid_q(y, lo[1], inv[1], nc[1]);
        const int qz = grid_q(z, lo[2], inv[2], nc[2]);
        return (qz * nc[1] + qy) * nc[0] + qx;
    };
    // (3) histogram
    for (int k = tid; k < n; k += T)
        atomicAdd(&hist[cell_of(__ldg(xyz + 3 * k), __ldg(xyz + 3 * k + 1), __ldg(xyz + 3 * k + 2))], 1u);
    __syncthreads();
    // (4) exclusive scan (warp w owns kGridCells/32 consecutive cells) + largest cell population
    {
        constexpr int cpw = kGridCells / NW;
        uint32_t carry = 0u, mx = 0u;
        for (int c = warp * cpw + lane; c < (warp + 1) * cpw; c += 32) {
            const uint32_t v = hist[c];
            mx = max(mx, v);
            uint32_t inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += t;
            }
            hist[c] = carry + inc - v;
            carry += __shfl_sync(FULL, inc, 31);
        }
        mx = __reduce_max_sync(FULL, mx);
        if (lane == 0) { woff[warp] = carry; wmaxc[warp] = mx; }
        __syncthreads();
        if (warp == 0) {
            const uint32_t v = woff[lane];
            uint32_t inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += t;
            }
            woff[lane] = inc - v;
            wmaxc[lane] = __reduce_max_sync(FULL, wmaxc[lane]);
        }
        __syncthreads();
        const uint32_t off = woff[warp];
        for (int c = warp * cpw + lane; c < (warp + 1) * cpw; c += 32) {
            const uint32_t st = hist[c] + off;
            hist[c] = st;
            if (c <= ncell) cell_start[c] = (int)st;
        }
        if (tid == 0 && ncell == kGridCells) cell_start[kGridCells] = n;
    }
    ok = ok && wmaxc[0] <= (uint32_t)kMaxCell;
    if (tid == 0) {
        GridHdr h;
#pragma unroll
        for (int a = 0; a < 3; ++a) { h.lo[a] = lo[a]; h.inv[a] = inv[a]; h.n[a] = nc[a]; }
        h.ok = ok ? 1 : 0;
        *reinterpret_cast<GridHdr*>(hdr) = h;
    }
    if (!ok) return;  // uniform: this cloud goes to the brute-force kernel
    __syncthreads();
    // (5) scatter in arbitrary order inside a cell
    for (int k = tid; k < n; k += T) {
        const float x = __ldg(xyz + 3 * k), y = __ldg(xyz + 3 * k + 1), z = __ldg(xyz + 3 * k + 2);
        const uint32_t pos = atomicAdd(&hist[cell_of(x, y, z)], 1u);
        tmp[pos] = make_float4(x, y, z, __int_as_float(k));
    }
    __syncthreads();  // tmp[] of this CTA is visible to it; hist[c] is now the END of cell c
    // (6) ascending original index inside every cell
    for (int p = tid; p < n; p += T) {
        const float4 e = tmp[p];
        const int c = cell_of(e.x, e.y, e.z);
        const int beg = c > 0 ? (int)hist[c - 1] : 0, end = (int)hist[c];
        const int me = __float_as_int(e.w);
        int before = 0;
        for (int j = beg; j < end; ++j) before += (__float_as_int(tmp[j].w) < me) ? 1 : 0;
        sorted[beg + before] = e;
    }
}

__global__ void __launch_bounds__(1024, 1)
    bq_grid_build_kernel(int n, float rout, const float* __restrict__ xyz_all, int* __restrict__ hdr_all,
                         int* __restrict__ cell_start_all, float4* sorted_tmp_all, float4* __restrict__ sorted_all) {
    const int cloud = blockIdx.x;
    grid_build_cloud(n, rout, xyz_all + (size_t)cloud * n * 3, hdr_all + (size_t)cloud * kHdrInts,
                     cell_start_all + (size_t)cloud * (kGridCells + 1), sorted_tmp_all + (size_t)cloud * n,
                     sorted_all + (size_t)cloud * n);
}

// Stacked clouds: frame f holds points start[f] .. start[f+1]-1 of xyz (N,3); its sorted records carry frame-local
// indices.
__global__ void __launch_bounds__(1024, 1)
    bq_grid_build_ragged_kernel(float rout, const int* __restrict__ start, const float* __restrict__ xyz,
                                int* __restrict__ hdr_all, int* __restrict__ cell_start_all, float4* sorted_tmp,
                                float4* __restrict__ sorted) {
    const int f = blockIdx.x;
    const int s = start[f];
    grid_build_cloud(start[f + 1] - s, rout, xyz + (size_t)s * 3, hdr_all + (size_t)f * kHdrInts,
                     cell_start_all + (size_t)f * (kGridCells + 1), sorted_tmp + s, sorted + s);
}

// The `nsample` smallest hit indices (ascending) of the centre (cx, cy, cz) in one cloud's grid, written to row[0..cnt)
// as index + off by the lanes that own them; returns cnt.  Lane l < 27 walks the sorted list of one neighbour cell up
// to its next hit; the warp repeatedly takes the smallest pending index (redux.sync.min).
template <bool DILATED>
__device__ __forceinline__ int grid_merge_core(int lane, const GridHdr& h, const int* __restrict__ cell_start,
                                               const float4* __restrict__ sorted, float cx, float cy, float cz, float rin2,
                                               float rout2, int nsample, int* const row, int off) {
    // lane l < 27 owns neighbour cell (dz, dy, dx) = (l / 9 - 1, l / 3 % 3 - 1, l % 3 - 1)
    int head = 0, end = 0;
    if (lane < 27) {
        const int gx = grid_q(cx, h.lo[0], h.inv[0], h.n[0]) + lane % 3 - 1;
        const int gy = grid_q(cy, h.lo[1], h.inv[1], h.n[1]) + (lane / 3) % 3 - 1;
        const int gz = grid_q(cz, h.lo[2], h.inv[2], h.n[2]) + lane / 9 - 1;
        if (gx >= 0 && gx < h.n[0] && gy >= 0 && gy < h.n[1] && gz >= 0 && gz < h.n[2]) {
            const int c = (gz * h.n[1] + gy) * h.n[0] + gx;
            head = __ldg(cell_start + c);
            end = __ldg(cell_start + c + 1);
        }
    }
    // cur = the lane's next hit in its (index-sorted) cell, or "none"
    uint32_t cur = 0xffffffffu;
    auto advance = [&]() {
        cur = 0xffffffffu;
        while (head < end) {
            const float4 p = sorted[head];
            ++head;
            const float d2 = sqdist3(p.x, p.y, p.z, cx, cy, cz);
            const bool hit = DILATED ? (d2 >= rin2 && d2 < rout2) : (d2 < rout2);
            if (hit) {
                cur = (uint32_t)__float_as_int(p.w);
                break;
            }
        }
    };
    advance();
    int cnt = 0;
    while (cnt < nsample) {
        const uint32_t mn = __reduce_min_sync(FULL, cur);
        if (mn == 0xffffffffu) break;
        if (cur == mn) {
            row[cnt] = (int)mn + off;
            advance();
        }
        ++cnt;
    }
    return cnt;
}

template <bool DILATED>
__global__ void __launch_bounds__(256)
    bq_grid_merge_kernel(int b, int n, int m, float rin2, float rout2, int nsample, const float* __restrict__ new_xyz,
                         const int* __restrict__ hdr_all, const int* __restrict__ cell_start_all,
                         const float4* __restrict__ sorted_all, int* __restrict__ idx_cnt, int* __restrict__ idx) {
    const int lane = threadIdx.x & 31;
    const long long wid = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (wid >= (long long)b * m) return;
    const int cloud = (int)(wid / m);
    const GridHdr h = *reinterpret_cast<const GridHdr*>(hdr_all + (size_t)cloud * kHdrInts);
    if (!h.ok) return;
    const int* __restrict__ cell_start = cell_start_all + (size_t)cloud * (kGridCells + 1);
    const float4* __restrict__ sorted = sorted_all + (size_t)cloud * n;
    const float* q = new_xyz + (size_t)wid * 3;
    const float cx = __ldg(q), cy = __ldg(q + 1), cz = __ldg(q + 2);
    int* const row = idx + (size_t)wid * nsample;

    const int cnt = grid_merge_core<DILATED>(lane, h, cell_start, sorted, cx, cy, cz, rin2, rout2, nsample, row, 0);
    // counts + cyclic padding (row[p] = row[p mod cnt]); rows without hits are zeroed
    __syncwarp();
    if (lane == 0) idx_cnt[wid] = cnt;
    if (cnt == 0) {
        for (int p = lane; p < nsample; p += 32) row[p] = 0;
    } else if (cnt < nsample) {
        for (int p = cnt + lane; p < nsample; p += 32) row[p] = row[p % cnt];
    }
}

// The half-warp search of bq_grid_query16_kernel for the centre (cx, cy, cz) in one cloud's grid: lane e of the half
// ends with the (e + 16 i)-th smallest hit index in best[i] (NONE past the last); returns the number of hits kept
// (<= nsample).  CANDIDATE-parallel: the candidates of the 27 cells are numbered 0..C-1 (prefix sum over the lanes' cell
// populations); in super-rounds of 64 every lane loads four of them at once (independent loads: one L2 round trip per
// 64 candidates instead of one per emitted hit), keeps the hits, and the half-warp extracts the smallest pending indices
// with redux.sync.min.  The kept hits re-enter the next super-round as pending values, so the result is the nsample
// smallest indices overall.
template <bool DILATED, int R>
__device__ __forceinline__ int grid_query16_core(int gl, unsigned gmask, const GridHdr& h, const int* __restrict__ cell_start,
                                                 const float4* __restrict__ sorted, float cx, float cy, float cz, float rin2,
                                                 float rout2, int nsample, uint32_t (&best)[R]) {
    constexpr int K = 4;
    constexpr uint32_t NONE = 0xffffffffu;
    const int qx = grid_q(cx, h.lo[0], h.inv[0], h.n[0]), qy = grid_q(cy, h.lo[1], h.inv[1], h.n[1]),
              qz = grid_q(cz, h.lo[2], h.inv[2], h.n[2]);
    int beg[2] = {0, 0}, len[2] = {0, 0};
#pragma unroll
    for (int s = 0; s < 2; ++s) {
        const int ci = gl + 16 * s;  // neighbour cell (dz, dy, dx) = (ci / 9 - 1, ci / 3 % 3 - 1, ci % 3 - 1)
        const int gx = qx + ci % 3 - 1, gy = qy + (ci / 3) % 3 - 1, gz = qz + ci / 9 - 1;
        if (ci < 27 && gx >= 0 && gx < h.n[0] && gy >= 0 && gy < h.n[1] && gz >= 0 && gz < h.n[2]) {
            const int c = (gz * h.n[1] + gy) * h.n[0] + gx;
            beg[s] = __ldg(cell_start + c);
            len[s] = __ldg(cell_start + c + 1) - beg[s];
        }
    }
    const int loc = len[0] + len[1];
    int incl = loc;  // inclusive prefix of the lanes' candidate counts within the half-warp
#pragma unroll
    for (int o = 1; o < 16; o <<= 1) {
        const int t = __shfl_up_sync(gmask, incl, o, 16);
        if (gl >= o) incl += t;
    }
    const int total = __shfl_sync(gmask, incl, 15, 16);
    const int excl_len0 = ((incl - loc) << 16) | len[0];  // (both < 2^15: a cell holds <= kMaxCell points, 27 cells)

    // lane e of the half: the (e + 16 i)-th smallest hit so far
#pragma unroll
    for (int i = 0; i < R; ++i) best[i] = NONE;
    for (int base = 0; base < total; base += 16 * K) {
        uint32_t v[K + R];
#pragma unroll
        for (int k = 0; k < K; ++k) {
            v[k] = NONE;
            if (base + k * 16 >= total) continue;  // (uniform in the half) no candidates left for this slot
            const int j = base + k * 16 + gl;
            int t = 0;  // owner lane = first lane whose inclusive prefix exceeds j
#pragma unroll
            for (int step = 8; step > 0; step >>= 1) {
                const int val = __shfl_sync(gmask, incl, t + step - 1, 16);
                if (val <= j) t += step;
            }
            t &= 15;
            const int el = __shfl_sync(gmask, excl_len0, t, 16);
            const int b0 = __shfl_sync(gmask, beg[0], t, 16), b1 = __shfl_sync(gmask, beg[1], t, 16);
            const int jj = j - (el >> 16), l0 = el & 0xffff;
            const int src = jj < l0 ? b0 + jj : b1 + (jj - l0);
            if (j < total) {
                const float4 p = sorted[src];
                const float d2 = sqdist3(p.x, p.y, p.z, cx, cy, cz);
                const bool hit = DILATED ? (d2 >= rin2 && d2 < rout2) : (d2 < rout2);
                if (hit) v[k] = (uint32_t)__float_as_int(p.w);
            }
        }
#pragma unroll
        for (int i = 0; i < R; ++i) v[K + i] = best[i];
        uint32_t nb[R];
#pragma unroll
        for (int i = 0; i < R; ++i) nb[i] = NONE;
        for (int e = 0; e < nsample; ++e) {
            uint32_t mine = v[0];
#pragma unroll
            for (int k = 1; k < K + R; ++k) mine = min(mine, v[k]);
            const uint32_t mn = __reduce_min_sync(gmask, mine);
            if (mn == NONE) break;
#pragma unroll
            for (int k = 0; k < K + R; ++k)
                if (v[k] == mn) v[k] = NONE;  // indices are unique: exactly one slot in the half-warp
#pragma unroll
            for (int i = 0; i < R; ++i)
                if (gl + 16 * i == e) nb[i] = mn;
        }
#pragma unroll
        for (int i = 0; i < R; ++i) best[i] = nb[i];
    }
    int cnt = 0;
#pragma unroll
    for (int i = 0; i < R; ++i) cnt += __popc(__ballot_sync(gmask, best[i] != NONE) & gmask);
    return cnt;
}

// nsample <= 16 * R (R = 1, 2): HALF a warp per centre (two centres per warp).  At the first SA layer a ball
// holds one or two points (the centre itself and maybe a neighbour) and a few dozen candidates, so a whole warp per centre
// is mostly fixed cost: ncu counts 346 warp-instructions per centre at 80 % issue utilisation -- the kernel is
// instruction-bound.  A lane owns neighbour cells gl and gl + 16 (candidates may be numbered in any order: the result is
// the nsample smallest hit indices whatever the order), collectives run on the half-warp's own member mask, lane e of the
// half ends up with the e-th (and, R = 2, the (e + 16)-th) smallest hit, and the grid is (centres, clouds) so that no
// 64-bit division is needed.
template <bool DILATED, int R>
__global__ void __launch_bounds__(256)
    bq_grid_query16_kernel(int n, int m, float rin2, float rout2, int nsample, const float* __restrict__ new_xyz,
                           const int* __restrict__ hdr_all, const int* __restrict__ cell_start_all,
                           const float4* __restrict__ sorted_all, int* __restrict__ idx_cnt, int* __restrict__ idx) {
    const int lane = threadIdx.x & 31, gl = lane & 15;
    const unsigned gmask = 0xffffu << (lane & 16);
    const int cloud = blockIdx.y;
    const int centre = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 2 + (lane >> 4);
    if (centre >= m) return;  // (a whole half-warp leaves together)
    const GridHdr h = *reinterpret_cast<const GridHdr*>(hdr_all + (size_t)cloud * kHdrInts);
    if (!h.ok) return;
    const int* __restrict__ cell_start = cell_start_all + (size_t)cloud * (kGridCells + 1);
    const float4* __restrict__ sorted = sorted_all + (size_t)cloud * n;
    const size_t wid = (size_t)cloud * m + centre;
    const float* q = new_xyz + wid * 3;
    const float cx = __ldg(q), cy = __ldg(q + 1), cz = __ldg(q + 2);
    int* const row = idx + wid * nsample;

    uint32_t best[R];
    const int cnt = grid_query16_core<DILATED, R>(gl, gmask, h, cell_start, sorted, cx, cy, cz, rin2, rout2, nsample, best);
    if (gl == 0) idx_cnt[wid] = cnt;
    // row[p] = hit[p mod cnt] (cyclic padding); rows without hits are zeroed
#pragma unroll
    for (int i = 0; i < R; ++i) {
        const int p = gl + 16 * i;
        const int src = cnt > 1 ? p % cnt : 0;
        uint32_t val = __shfl_sync(gmask, best[0], src & 15, 16);
        if (R > 1) {
            const uint32_t hi = __shfl_sync(gmask, best[R - 1], src & 15, 16);
            if (src >= 16) val = hi;
        }
        if (p < nsample) row[p] = cnt ? (int)val : 0;
    }
}

// ---- stacked (ragged) clouds, pointnet2_stack's ball_query_kernel_stack contract: centre p belongs to frame
// stack_frame_of(p); its row holds the first min(hits, nsample) frame-local hit indices in ascending order, the
// remaining slots repeat the FIRST hit, and a row without hits gets only row[0] = -1 (the caller zeroed the rest).
// global_rows != 0 (the fused SA path): frame start + index instead, and all-zero rows without hits.  idx_cnt may be
// null.  Frames whose grid is unusable are left to stack_ball_query_kernel (ball_query.cu).
template <int R>
__global__ void __launch_bounds__(256)
    bq_grid_query16_ragged_kernel(int b, int m, float rout2, int nsample, const float* __restrict__ new_xyz,
                                  const int* __restrict__ mstart, const int* __restrict__ nstart,
                                  const int* __restrict__ hdr_all, const int* __restrict__ cell_start_all,
                                  const float4* __restrict__ sorted_all, int* __restrict__ idx_cnt, int* __restrict__ idx,
                                  int global_rows) {
    const int lane = threadIdx.x & 31, gl = lane & 15;
    const unsigned gmask = 0xffffu << (lane & 16);
    const int centre = (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5)) * 2 + (lane >> 4);
    if (centre >= m) return;  // (a whole half-warp leaves together)
    const int f = stack_frame_of(centre, b, mstart);
    const GridHdr h = *reinterpret_cast<const GridHdr*>(hdr_all + (size_t)f * kHdrInts);
    if (!h.ok) return;
    const int start = __ldg(nstart + f);
    const float* q = new_xyz + (size_t)centre * 3;
    const float cx = __ldg(q), cy = __ldg(q + 1), cz = __ldg(q + 2);
    int* const row = idx + (size_t)centre * nsample;

    uint32_t best[R];
    const int cnt = grid_query16_core<false, R>(gl, gmask, h, cell_start_all + (size_t)f * (kGridCells + 1),
                                                sorted_all + start, cx, cy, cz, 0.f, rout2, nsample, best);
    if (idx_cnt && gl == 0) idx_cnt[centre] = cnt;
    const int off = global_rows ? start : 0;
#pragma unroll
    for (int i = 0; i < R; ++i) {
        const int p = gl + 16 * i;
        const int src = p < cnt ? p : 0;  // past the hits: the first hit
        uint32_t val = __shfl_sync(gmask, best[0], src & 15, 16);
        if (R > 1) {
            const uint32_t hi = __shfl_sync(gmask, best[R - 1], src & 15, 16);
            if (src >= 16) val = hi;
        }
        if (p < nsample) {
            if (cnt) row[p] = (int)val + off;
            else if (global_rows) row[p] = 0;
            else if (p == 0) row[0] = -1;
        }
    }
}

// nsample > 32: one warp per centre (the merge walk of bq_grid_merge_kernel), same contract as above.
__global__ void __launch_bounds__(256)
    bq_grid_merge_ragged_kernel(int b, int m, float rout2, int nsample, const float* __restrict__ new_xyz,
                                const int* __restrict__ mstart, const int* __restrict__ nstart,
                                const int* __restrict__ hdr_all, const int* __restrict__ cell_start_all,
                                const float4* __restrict__ sorted_all, int* __restrict__ idx_cnt, int* __restrict__ idx,
                                int global_rows) {
    const int lane = threadIdx.x & 31;
    const int centre = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (centre >= m) return;
    const int f = stack_frame_of(centre, b, mstart);
    const GridHdr h = *reinterpret_cast<const GridHdr*>(hdr_all + (size_t)f * kHdrInts);
    if (!h.ok) return;
    const int start = __ldg(nstart + f);
    const float* q = new_xyz + (size_t)centre * 3;
    const float cx = __ldg(q), cy = __ldg(q + 1), cz = __ldg(q + 2);
    int* const row = idx + (size_t)centre * nsample;
    const int off = global_rows ? start : 0;

    const int cnt = grid_merge_core<false>(lane, h, cell_start_all + (size_t)f * (kGridCells + 1), sorted_all + start,
                                           cx, cy, cz, 0.f, rout2, nsample, row, off);
    __syncwarp();  // row[0] (the first hit) was written by whichever lane owned it
    if (idx_cnt && lane == 0) idx_cnt[centre] = cnt;
    if (cnt == 0) {
        if (global_rows)
            for (int p = lane; p < nsample; p += 32) row[p] = 0;
        else if (lane == 0)
            row[0] = -1;
    } else {
        const int first = row[0];
        for (int p = cnt + lane; p < nsample; p += 32) row[p] = first;
    }
}

constexpr int kBuildSmem = kGridCells * sizeof(uint32_t);  // the build's shared-memory histogram

// The grids of b clouds holding npts points in all, carved from scratch buffer `tag`: the headers, the cell starts and
// the scattered / index-sorted point records, each array 256-byte aligned.
struct GridScratch {
    int* hdr;
    int* cell_start;
    float4* tmp;
    float4* sorted;
};

static int grid_scratch(int tag, int b, size_t npts, cudaStream_t stream, GridScratch* g) {
    auto align = [](size_t bytes) { return (bytes + 255) & ~(size_t)255; };
    const size_t hdr_bytes = align((size_t)b * kHdrInts * sizeof(int));
    const size_t cs_bytes = align((size_t)b * (kGridCells + 1) * sizeof(int));
    const size_t pts_bytes = align(npts * sizeof(float4));
    void* base = nullptr;
    const int rc = tsm_scratch_get(tag, hdr_bytes + cs_bytes + 2 * pts_bytes, stream, &base);
    if (rc != TSM_OK) return rc;
    unsigned char* const p = static_cast<unsigned char*>(base);
    g->hdr = reinterpret_cast<int*>(p);
    g->cell_start = reinterpret_cast<int*>(p + hdr_bytes);
    g->tmp = reinterpret_cast<float4*>(p + hdr_bytes + cs_bytes);
    g->sorted = reinterpret_cast<float4*>(p + hdr_bytes + cs_bytes + pts_bytes);
    return TSM_OK;
}

}  // namespace tsm

int tsm_grid_build(int b, int n, float rout, const float* xyz, cudaStream_t stream, int tag, const int** hdr_out,
                   const int** cell_start_out, const float4** sorted_out) {
    using namespace tsm;
    GridScratch g;
    const int rc = grid_scratch(tag, b, (size_t)b * n, stream, &g);
    if (rc != TSM_OK) return rc;
    TSM_CUDA_TRY(cudaFuncSetAttribute(bq_grid_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBuildSmem));
    bq_grid_build_kernel<<<b, 1024, kBuildSmem, stream>>>(n, rout, xyz, g.hdr, g.cell_start, g.tmp, g.sorted);
    TSM_LAUNCH_CHECK();
    *hdr_out = g.hdr;
    *cell_start_out = g.cell_start;
    *sorted_out = g.sorted;
    return TSM_OK;
}

// Builds the grids of all clouds and answers every cloud whose grid is usable.  *grid_hdr receives the
// per-cloud header array (device; int [b][16], word 9 = usable) for the brute-force kernel to consult.
int tsm_ball_query_grid(bool dilated, int b, int n, int m, float rin, float rout, int nsample, const float* new_xyz,
                        const float* xyz, int* idx_cnt, int* idx, cudaStream_t stream, const int** grid_hdr) {
    using namespace tsm;
    const int *hdr = nullptr, *cell_start = nullptr;
    const float4* sorted = nullptr;
    if (!(rout > 0.f)) {  // no ball: nothing can hit; leave every cloud to the brute-force kernel
        *grid_hdr = nullptr;
        return TSM_OK;
    }
    int rc = tsm_grid_build(b, n, rout, xyz, stream, 4, &hdr, &cell_start, &sorted);
    if (rc != TSM_OK) return rc;
    const float rin2 = rin * rin, rout2 = rout * rout;  // f32 products, as ball_query_gpu.cu:91, 154-155
    if (nsample <= 32) {
        const dim3 grid16((unsigned)((m + 15) / 16), (unsigned)b);
#define BQ16(D, RR) bq_grid_query16_kernel<D, RR><<<grid16, 256, 0, stream>>>(n, m, rin2, rout2, nsample, new_xyz, hdr, cell_start, sorted, idx_cnt, idx)
        if (nsample <= 16) {
            if (dilated) BQ16(true, 1); else BQ16(false, 1);
        } else {
            if (dilated) BQ16(true, 2); else BQ16(false, 2);
        }
#undef BQ16
    } else {
        const unsigned blocks = (unsigned)(((long long)b * m + 7) / 8);
        if (dilated)
            bq_grid_merge_kernel<true><<<blocks, 256, 0, stream>>>(b, n, m, rin2, rout2, nsample, new_xyz, hdr,
                                                                   cell_start, sorted, idx_cnt, idx);
        else
            bq_grid_merge_kernel<false><<<blocks, 256, 0, stream>>>(b, n, m, rin2, rout2, nsample, new_xyz, hdr,
                                                                    cell_start, sorted, idx_cnt, idx);
    }
    TSM_LAUNCH_CHECK();
    *grid_hdr = hdr;
    return TSM_OK;
}

int tsm_grid_build_ragged(int b, int n_total, float rout, const int* start, const float* xyz, cudaStream_t stream, int tag,
                          const int** hdr_out, const int** cell_start_out, const float4** sorted_out) {
    using namespace tsm;
    GridScratch g;
    const int rc = grid_scratch(tag, b, (size_t)n_total, stream, &g);
    if (rc != TSM_OK) return rc;
    TSM_CUDA_TRY(cudaFuncSetAttribute(bq_grid_build_ragged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBuildSmem));
    bq_grid_build_ragged_kernel<<<b, 1024, kBuildSmem, stream>>>(rout, start, xyz, g.hdr, g.cell_start, g.tmp, g.sorted);
    TSM_LAUNCH_CHECK();
    *hdr_out = g.hdr;
    *cell_start_out = g.cell_start;
    *sorted_out = g.sorted;
    return TSM_OK;
}

int tsm_stack_ball_query_grid(int b, int m, int n_total, float radius, int nsample, const float* new_xyz,
                              const int* mstart, const int* nstart, const float* xyz, int* idx, int* idx_cnt,
                              int global_rows, cudaStream_t stream, const int** grid_hdr) {
    using namespace tsm;
    *grid_hdr = nullptr;
    // radius * radius is what the query compares: a negative radius is its absolute value, 0 / NaN hit nothing (every
    // frame then goes to the brute-force kernel)
    const float rout = fabsf(radius);
    if (!(rout > 0.f) || n_total <= 0) return TSM_OK;
    const int *hdr = nullptr, *cell_start = nullptr;
    const float4* sorted = nullptr;
    const int rc = tsm_grid_build_ragged(b, n_total, rout, nstart, xyz, stream, 9, &hdr, &cell_start, &sorted);
    if (rc != TSM_OK) return rc;
    const float rout2 = radius * radius;  // f32 product, as ball_query_gpu.cu (stack):25
    if (nsample <= 32) {
        const unsigned blocks = (unsigned)((m + 15) / 16);
        if (nsample <= 16)
            bq_grid_query16_ragged_kernel<1><<<blocks, 256, 0, stream>>>(b, m, rout2, nsample, new_xyz, mstart, nstart, hdr,
                                                                         cell_start, sorted, idx_cnt, idx, global_rows);
        else
            bq_grid_query16_ragged_kernel<2><<<blocks, 256, 0, stream>>>(b, m, rout2, nsample, new_xyz, mstart, nstart, hdr,
                                                                         cell_start, sorted, idx_cnt, idx, global_rows);
    } else {
        bq_grid_merge_ragged_kernel<<<(unsigned)((m + 7) / 8), 256, 0, stream>>>(b, m, rout2, nsample, new_xyz, mstart, nstart,
                                                                                 hdr, cell_start, sorted, idx_cnt, idx,
                                                                                 global_rows);
    }
    TSM_LAUNCH_CHECK();
    *grid_hdr = hdr;
    return TSM_OK;
}
