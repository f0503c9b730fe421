// roiaware_pool3d.cu -- the roiaware_pool3d ops (PartA2's RoI pooling and every point head's target assignment):
// points_in_boxes_gpu, points_in_boxes_cpu (host code), RoIAwarePool3d forward and backward (sm_100a).
//
// Replaces (same labels, lists, argmax and pooled values, bit for bit, as far as the recalled contract below is the
// reference's; gradients up to the order of the atomic adds):
//   points_in_boxes_kernel, generate_pts_mask_for_box3d + collect_inside_pts_for_box3d, roiaware_maxpool3d /
//   roiaware_avgpool3d and their backward kernels, points_in_boxes_cpu
//   (upstream OpenPCDet roiaware_pool3d/src/roiaware_pool3d_kernel.cu, roiaware_pool3d.cpp)
//
// Contract (restated from upstream OpenPCDet; every item is RECALLED, not read: the reference tree was not available
// where this was written -- the head-to-head test settles it where the reference is built):
//   * box [cx, cy, cz, dx, dy, dz, heading], (cx, cy, cz) the centre.  A point is inside iff
//       !(fabsf(z - cz) > dz / 2.0)                                     (double compare: z on the face is inside)
//       cosa = cosf(-heading), sina = sinf(-heading)                    (float, accurate cosf / sinf, no fast-math)
//       local_x = sx*cosa + sy*(-sina), local_y = sx*sina + sy*cosa,    sx = x - cx, sy = y - cy
//       fabs(local_x) < dx / 2.0 + MARGIN && fabs(local_y) < dy / 2.0 + MARGIN   (double compares)
//     MARGIN = 1e-5f on the GPU, 1e-2f in points_in_boxes_cpu.  On the GPU the products are contracted as nvcc 12.9
//     (-O3, default -fmad=true, sm_100a) contracts the recalled expressions -- checked in the SASS of a build of them:
//     local_x = fmaf(sx, cosa, -(sy*sina)), local_y = fmaf(sy, cosa, sx*sina).  The CPU form rounds every product
//     (x86-64 has no contraction without -mfma).
//   * Deviation, on purpose: a NaN coordinate (point or box) is never inside.  Upstream's `> dz / 2.0` form keeps a point
//     whose z - cz is NaN; here the z test is `<=`, so NaN fails it as it fails the x / y tests.
//   * points_in_boxes_gpu(boxes (B,T,7), pts (B,N,3), out (B,N)): out[b,n] = the FIRST k whose box holds the point; the
//     caller's pre-fill (-1) is left otherwise.  points_in_boxes_cpu(boxes (M,7), pts (N,3), out (M,N)): 0 / 1 per pair.
//   * forward(rois (R,7), pts (P,3), pts_feature (P,C), argmax (R,X,Y,Z,C), pts_idx_of_voxels (R,X,Y,Z,L), pooled
//     (R,X,Y,Z,C), pool_method 0 max / 1 avg); X, Y, Z from argmax's shape, L from dim 4 of pts_idx_of_voxels, every
//     output dimension <= 256 (the voxel code packs x, y, z in 8 bits each).  For an inside point
//       local_z = z - cz, x_res = dx / X (float), x_idx = (unsigned) int((local_x + dx / 2) / x_res), the int conversion
//       being cvt.rzi.s32.f32 (NaN -> 0, saturating at +-inf), then the UNSIGNED min(max(x_idx, 0), X - 1): a negative
//       index lands in the last voxel.  Same for y and z.
//     Slot 0 of a voxel's list is its counter; points are appended in ascending point index while counter < L - 1, so
//     the counter saturates at L - 1.  Max pool: max_val = -1e50 (-inf in float), argmax = -1, strict > over the list in
//     order (the first maximum wins; NaN and -inf are never taken), pooled written only when argmax != -1, argmax always.
//     Avg pool: float sum in list order, pooled = sum / count written only when count > 0, argmax not written.
//   * backward(pts_idx_of_voxels, argmax, grad_out (R,X,Y,Z,C), grad_in (P,C), pool_method): max: grad_in[argmax, c] +=
//     grad_out * 1 where argmax != -1; avg: grad_in[pt, c] += grad_out * (1 / fmaxf(count, 1)) for every listed point.
//     Float atomics, as upstream.
//
// Design:
//  * points_in_boxes: one CTA per (frame, 256 points); the frame's boxes are staged in shared memory 1024 at a time with
//    cosf / sinf and the thresholds computed once per box (the same values a per-pair evaluation gives).  The double
//    thresholds become float ones with directed rounding, which decide every float exactly as the double compare does:
//    f < T  <=>  f < (T rounded up to float),  f <= D  <=>  f <= (D rounded down to float).  The CTA stops once every
//    one of its points has found a box.
//  * forward, lists: one CTA per RoI walks the points in index order, 1024 per tile; inside points are compacted in order
//    (ballot + a scan over the tile's 32 chunks) into a shared queue, and one warp appends the queue to the voxel lists,
//    32 entries at a time: __match_any_sync groups equal voxels, the rank among them keeps index order and the cap exact
//    without atomics.  The counters live in shared memory up to kRaSmemVoxels voxels per RoI, else in slot 0 of the
//    lists themselves (same lists).  The kernel writes every counter, so nothing depends on the caller's zero fill, and
//    there is no R x P mask and no allocation per call.
//  * forward, pooling / avg backward: a group of gw lanes per (RoI, voxel), gw = C rounded up to a power of two (<= 32),
//    lanes over channels, each lane walking the list in order -- the reference's tie rule and summation order exactly.
//  * 64-bit offsets wherever R*X*Y*Z*L or R*X*Y*Z*C can pass 2^31.
#include <math.h>
#include <string.h>

#include "common.cuh"

namespace tsm {

constexpr int kRaMaxOut = 256;          // the 8-bit fields of the voxel code
constexpr int kRaPibThreads = 256;
constexpr int kRaPibTile = 1024;        // boxes staged per pass (32 KB)
constexpr int kRaThreads = 256;         // list-build CTA
constexpr int kRaPerThread = 4;
constexpr int kRaTile = kRaThreads * kRaPerThread;  // points per tile
constexpr int kRaChunks = kRaTile / 32;             // 32-point chunks per tile, in point order
constexpr int kRaSmemVoxels = 16384;    // shared-memory counters up to this many voxels per RoI (64 KB)

// A box's test constants: (cx, cy, cz, cosa) and (sina, tx, ty, tz).  tx = dx / 2.0 + margin rounded up to float,
// tz = dz / 2.0 rounded down (a NaN stays NaN and fails every compare).
__device__ __forceinline__ void ra_box(const float* __restrict__ b, float margin, float4& p, float4& q) {
    const float h = __ldg(b + 6);
    p = make_float4(__ldg(b), __ldg(b + 1), __ldg(b + 2), cosf(-h));
    q = make_float4(sinf(-h), __double2float_ru((double)__ldg(b + 3) / 2.0 + (double)margin),
                    __double2float_ru((double)__ldg(b + 4) / 2.0 + (double)margin),
                    __double2float_rd((double)__ldg(b + 5) / 2.0));
}

// local_x / local_y with the reference's contraction (see the contract above)
__device__ __forceinline__ bool ra_inside(const float4& p, const float4& q, float x, float y, float z, float& lx,
                                          float& ly) {
    const float sx = __fsub_rn(x, p.x), sy = __fsub_rn(y, p.y);
    lx = __fmaf_rn(sx, p.w, __fmul_rn(sy, -q.x));
    ly = __fmaf_rn(sy, p.w, __fmul_rn(sx, q.x));
    return fabsf(__fsub_rn(z, p.z)) <= q.w && fabsf(lx) < q.y && fabsf(ly) < q.z;
}

// (unsigned) int((l + half) / res) with cvt.rzi.s32.f32, then the unsigned min(max(i, 0), n - 1)
__device__ __forceinline__ unsigned ra_cell(float l, float half, float res, int n) {
    const unsigned i = (unsigned)__float2int_rz(__fdiv_rn(__fadd_rn(l, half), res));
    return min(i, (unsigned)(n - 1));
}

__global__ void __launch_bounds__(kRaPibThreads)
    ra_points_in_boxes_kernel(int t, int n, const float* __restrict__ boxes, const float* __restrict__ pts,
                              int* __restrict__ out) {
    __shared__ float4 sp[kRaPibTile], sq[kRaPibTile];
    const int f = blockIdx.y;
    const int k = blockIdx.x * kRaPibThreads + threadIdx.x;
    boxes += (size_t)f * t * 7;
    float x = 0.f, y = 0.f, z = 0.f;
    bool done = k >= n;
    if (!done) {
        const float* const pt = pts + ((size_t)f * n + k) * 3;
        x = __ldg(pt); y = __ldg(pt + 1); z = __ldg(pt + 2);
    }
    for (int t0 = 0; t0 < t; t0 += kRaPibTile) {
        const int nt = min(kRaPibTile, t - t0);
        for (int j = threadIdx.x; j < nt; j += kRaPibThreads) ra_box(boxes + (size_t)(t0 + j) * 7, 1e-5f, sp[j], sq[j]);
        __syncthreads();
        if (!done) {
            for (int j = 0; j < nt; ++j) {
                float lx, ly;
                if (ra_inside(sp[j], sq[j], x, y, z, lx, ly)) {
                    out[(size_t)f * n + k] = t0 + j;
                    done = true;
                    break;
                }
            }
        }
        if (!__syncthreads_or(!done)) break;  // also keeps the tile until every thread is through it
    }
}

struct RaArgs {
    int r, p, c, X, Y, Z, L;
    const float* rois;
    const float* pts;
    const float* feats;
    int* idx;       // (R, X, Y, Z, L)
    int* argmax;    // (R, X, Y, Z, C)
    float* pooled;  // (R, X, Y, Z, C)
};

// The voxel lists of RoI blockIdx.x.  SMEM: the counters in shared memory, else in slot 0 of the lists.
template <bool SMEM>
__global__ void __launch_bounds__(kRaThreads) ra_lists_kernel(RaArgs a) {
    extern __shared__ int ra_cnt[];
    __shared__ int2 queue[kRaTile];  // (point, voxel) of the tile's inside points, ascending point
    __shared__ int chunk_off[kRaChunks + 1];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int V = a.X * a.Y * a.Z;
    const size_t L = (size_t)a.L;
    const int cap = a.L - 1;
    int* const lists = a.idx + (size_t)blockIdx.x * V * L;
    auto counter = [&](int v) -> int* { return SMEM ? ra_cnt + v : lists + (size_t)v * L; };
    for (int v = threadIdx.x; v < V; v += kRaThreads) *counter(v) = 0;

    const float* const roi = a.rois + (size_t)blockIdx.x * 7;
    float4 bp, bq;
    ra_box(roi, 1e-5f, bp, bq);
    const float dx = __ldg(roi + 3), dy = __ldg(roi + 4), dz = __ldg(roi + 5);
    const float hx = __fdiv_rn(dx, 2.f), hy = __fdiv_rn(dy, 2.f), hz = __fdiv_rn(dz, 2.f);
    const float rx = __fdiv_rn(dx, (float)a.X), ry = __fdiv_rn(dy, (float)a.Y), rz = __fdiv_rn(dz, (float)a.Z);
    const unsigned below = (1u << lane) - 1u;
    __syncthreads();

    for (int t0 = 0; t0 < a.p; t0 += kRaTile) {
        int code[kRaPerThread], rank[kRaPerThread];
#pragma unroll
        for (int j = 0; j < kRaPerThread; ++j) {
            const int k = t0 + j * kRaThreads + threadIdx.x;
            int v = -1;
            if (k < a.p) {
                const float* const pt = a.pts + (size_t)k * 3;
                const float x = __ldg(pt), y = __ldg(pt + 1), z = __ldg(pt + 2);
                float lx, ly;
                if (ra_inside(bp, bq, x, y, z, lx, ly)) {
                    const unsigned ix = ra_cell(lx, hx, rx, a.X), iy = ra_cell(ly, hy, ry, a.Y),
                                   iz = ra_cell(__fsub_rn(z, bp.z), hz, rz, a.Z);
                    v = (int)((ix * a.Y + iy) * a.Z + iz);
                }
            }
            code[j] = v;
            const unsigned bal = __ballot_sync(FULL, v >= 0);
            rank[j] = __popc(bal & below);
            if (lane == 0) chunk_off[j * (kRaThreads / 32) + warp] = __popc(bal);
        }
        __syncthreads();
        if (warp == 0) {  // exclusive scan of the chunk counts (chunk j * 8 + w = points t0 + 256 j + 32 w + lane)
            const int c = chunk_off[lane];
            int s = c;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int u = __shfl_up_sync(FULL, s, o);
                if (lane >= o) s += u;
            }
            chunk_off[lane] = s - c;
            if (lane == 31) chunk_off[kRaChunks] = s;
        }
        __syncthreads();
        const int total = chunk_off[kRaChunks];
        if (total == 0) continue;  // uniform: nothing of this tile is in the RoI
#pragma unroll
        for (int j = 0; j < kRaPerThread; ++j)
            if (code[j] >= 0)
                queue[chunk_off[j * (kRaThreads / 32) + warp] + rank[j]] =
                    make_int2(t0 + j * kRaThreads + threadIdx.x, code[j]);
        __syncthreads();
        if (warp == 0) {
            for (int q0 = 0; q0 < total; q0 += 32) {
                const bool has = q0 + lane < total;
                const int2 e = has ? queue[q0 + lane] : make_int2(0, -1);
                const unsigned peers = __match_any_sync(FULL, e.y);  // lanes without an entry group under -1
                int base = 0;
                if (has) base = *counter(e.y);
                __syncwarp();
                if (has) {
                    const int before = __popc(peers & below);
                    if (base + before < cap) lists[(size_t)e.y * L + 1 + base + before] = e.x;
                    if (before == 0) *counter(e.y) = min(base + __popc(peers), cap);
                }
                __syncwarp();
            }
        }
        __syncthreads();
    }
    if (SMEM)
        for (int v = threadIdx.x; v < V; v += kRaThreads) lists[(size_t)v * L] = ra_cnt[v];
}

// The valid part of list `g`: its counter clamped to [0, L - 1] (the forward never writes more; a caller's tensor may)
__device__ __forceinline__ int ra_list_len(const int* list, int L) { return min(max(__ldg(list), 0), L - 1); }

// Max / avg pooling: a group of 1 << gw_log2 lanes per (RoI, voxel) g, lanes over channels.
template <bool AVG>
__global__ void __launch_bounds__(256) ra_pool_kernel(RaArgs a, int gw_log2, long long groups) {
    const int gw = 1 << gw_log2;
    const int c0 = threadIdx.x & (gw - 1);
    const float ninf = __int_as_float(0xff800000);
    for (long long g = ((long long)blockIdx.x * 256 + threadIdx.x) >> gw_log2; g < groups;
         g += ((long long)gridDim.x * 256) >> gw_log2) {
        const int* const list = a.idx + g * a.L;
        const int n = ra_list_len(list, a.L);
        for (int ch = c0; ch < a.c; ch += gw) {
            if (AVG) {
                if (n == 0) break;  // an empty voxel keeps the caller's zeros
                float s = 0.f;
                for (int k = 1; k <= n; ++k) {
                    const int pt = __ldg(list + k);
                    if ((unsigned)pt < (unsigned)a.p) s = __fadd_rn(s, __ldg(a.feats + (size_t)pt * a.c + ch));
                }
                a.pooled[g * a.c + ch] = __fdiv_rn(s, (float)n);
            } else {
                float best = ninf;
                int arg = -1;
                for (int k = 1; k <= n; ++k) {
                    const int pt = __ldg(list + k);
                    if ((unsigned)pt >= (unsigned)a.p) continue;
                    const float v = __ldg(a.feats + (size_t)pt * a.c + ch);
                    if (v > best) { best = v; arg = pt; }
                }
                if (arg != -1) a.pooled[g * a.c + ch] = best;
                a.argmax[g * a.c + ch] = arg;
            }
        }
    }
}

// Max backward: grad_in[argmax[e], c] += grad_out[e] for every element e = (RoI, voxel, c) with argmax[e] in [0, P).
__global__ void __launch_bounds__(256) ra_max_grad_kernel(long long work, int c, int p, const int* __restrict__ argmax,
                                                          const float* __restrict__ grad_out, float* __restrict__ grad_in) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < work; e += (long long)gridDim.x * 256) {
        const int k = __ldg(argmax + e);
        if ((unsigned)k < (unsigned)p) atomicAdd(grad_in + (size_t)k * c + (int)(e % c), __ldg(grad_out + e));
    }
}

// Avg backward: grad_in[pt, c] += grad_out[g, c] * (1 / fmaxf(count, 1)) for every listed point pt of voxel group g.
__global__ void __launch_bounds__(256)
    ra_avg_grad_kernel(long long groups, int gw_log2, int c, int p, int L, const int* __restrict__ idx,
                       const float* __restrict__ grad_out, float* __restrict__ grad_in) {
    const int gw = 1 << gw_log2;
    const int c0 = threadIdx.x & (gw - 1);
    for (long long g = ((long long)blockIdx.x * 256 + threadIdx.x) >> gw_log2; g < groups;
         g += ((long long)gridDim.x * 256) >> gw_log2) {
        const int* const list = idx + g * L;
        const int n = ra_list_len(list, L);
        if (n == 0) continue;
        const float w = __fdiv_rn(1.f, fmaxf((float)n, 1.f));
        for (int ch = c0; ch < c; ch += gw) {
            const float t = __fmul_rn(__ldg(grad_out + g * c + ch), w);
            for (int k = 1; k <= n; ++k) {
                const int pt = __ldg(list + k);
                if ((unsigned)pt < (unsigned)p) atomicAdd(grad_in + (size_t)pt * c + ch, t);
            }
        }
    }
}

static bool ra_dims_ok(int r, int p, int c, int X, int Y, int Z, int L) {
    return r >= 0 && p >= 0 && c >= 0 && X >= 1 && X <= kRaMaxOut && Y >= 1 && Y <= kRaMaxOut && Z >= 1 &&
           Z <= kRaMaxOut && L >= 1;
}

static int ra_group_log2(int c) {
    int l = 0;
    while (l < 5 && (1 << l) < c) ++l;
    return l;
}

static unsigned ra_blocks(long long threads) {
    const long long want = (threads + 255) / 256, cap = (long long)tsm_num_sms() * 32;
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace tsm

// Host code of points_in_boxes_cpu (MARGIN 1e-2f).  Every product is rounded on its own (ra_rn), so no compiler
// contraction can change a label.
static float ra_rn(float v) {
    volatile float t = v;
    return t;
}

extern "C" {

int tsmdet_points_in_boxes(int b, int t, int n, const float* boxes, const float* pts, int* box_idx_of_points,
                           void* stream) {
    using namespace tsm;
    if (b < 0 || t < 0 || n < 0) return TSM_ERR_INVALID;
    if (b == 0 || t == 0 || n == 0) return TSM_OK;
    if (!boxes || !pts || !box_idx_of_points || b > 65535) return TSM_ERR_INVALID;
    const dim3 grid((unsigned)divup(n, kRaPibThreads), (unsigned)b);
    ra_points_in_boxes_kernel<<<grid, kRaPibThreads, 0, (cudaStream_t)stream>>>(t, n, boxes, pts, box_idx_of_points);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_points_in_boxes_cpu(int m, int n, const float* boxes, const float* pts, int* pts_indices) {
    if (m < 0 || n < 0) return TSM_ERR_INVALID;
    if (m == 0 || n == 0) return TSM_OK;
    if (!boxes || !pts || !pts_indices) return TSM_ERR_INVALID;
    const float margin = 1e-2f;
    for (int i = 0; i < m; ++i) {
        const float* const bx = boxes + (size_t)i * 7;
        const float cosa = cosf(-bx[6]), sina = sinf(-bx[6]);
        const double tx = bx[3] / 2.0 + margin, ty = bx[4] / 2.0 + margin, tz = bx[5] / 2.0;
        for (int j = 0; j < n; ++j) {
            const float* const pt = pts + (size_t)j * 3;
            const float sx = pt[0] - bx[0], sy = pt[1] - bx[1];
            const float lx = ra_rn(sx * cosa) + ra_rn(sy * -sina);
            const float ly = ra_rn(sx * sina) + ra_rn(sy * cosa);
            pts_indices[(size_t)i * n + j] = fabsf(pt[2] - bx[2]) <= tz && fabs(lx) < tx && fabs(ly) < ty;
        }
    }
    return TSM_OK;
}

int tsmdet_roiaware_pool3d(int r, int p, int c, int out_x, int out_y, int out_z, int max_pts_each_voxel,
                           const float* rois, const float* pts, const float* pts_feature, int* argmax,
                           int* pts_idx_of_voxels, float* pooled_features, int pool_method, void* stream_) {
    using namespace tsm;
    if (!ra_dims_ok(r, p, c, out_x, out_y, out_z, max_pts_each_voxel) || (pool_method != 0 && pool_method != 1))
        return TSM_ERR_INVALID;
    if (r == 0) return TSM_OK;
    if (!rois || !pts_idx_of_voxels || (p > 0 && !pts) || (c > 0 && (!argmax || !pooled_features)) ||
        (p > 0 && c > 0 && !pts_feature))
        return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    RaArgs a = {r, p, c, out_x, out_y, out_z, max_pts_each_voxel, rois, pts, pts_feature, pts_idx_of_voxels, argmax,
                pooled_features};
    const int V = out_x * out_y * out_z;
    if (V <= kRaSmemVoxels) {
        const int smem = V * (int)sizeof(int);
        TSM_CUDA_TRY(cudaFuncSetAttribute(ra_lists_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        ra_lists_kernel<true><<<(unsigned)r, kRaThreads, smem, stream>>>(a);
    } else {
        ra_lists_kernel<false><<<(unsigned)r, kRaThreads, 0, stream>>>(a);
    }
    TSM_LAUNCH_CHECK();
    if (c == 0) return TSM_OK;
    const long long groups = (long long)r * V;
    const int gl = ra_group_log2(c);
    if (pool_method == 0)
        ra_pool_kernel<false><<<ra_blocks(groups << gl), 256, 0, stream>>>(a, gl, groups);
    else
        ra_pool_kernel<true><<<ra_blocks(groups << gl), 256, 0, stream>>>(a, gl, groups);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_roiaware_pool3d_grad(int r, int p, int c, int out_x, int out_y, int out_z, int max_pts_each_voxel,
                                const int* pts_idx_of_voxels, const int* argmax, const float* grad_out, float* grad_in,
                                int pool_method, void* stream_) {
    using namespace tsm;
    if (!ra_dims_ok(r, p, c, out_x, out_y, out_z, max_pts_each_voxel) || (pool_method != 0 && pool_method != 1))
        return TSM_ERR_INVALID;
    if (r == 0 || p == 0 || c == 0) return TSM_OK;
    if (!grad_out || !grad_in || (pool_method == 0 ? !argmax : !pts_idx_of_voxels)) return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    const long long groups = (long long)r * out_x * out_y * out_z;
    if (pool_method == 0) {
        ra_max_grad_kernel<<<ra_blocks(groups * c), 256, 0, stream>>>(groups * c, c, p, argmax, grad_out, grad_in);
    } else {
        const int gl = ra_group_log2(c);
        ra_avg_grad_kernel<<<ra_blocks(groups << gl), 256, 0, stream>>>(groups, gl, c, p, max_pts_each_voxel,
                                                                        pts_idx_of_voxels, grad_out, grad_in);
    }
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

}  // extern "C"
