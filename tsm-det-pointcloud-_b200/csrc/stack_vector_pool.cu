// stack_vector_pool.cu -- the vector-pool ops of pointnet2_stack (PV-RCNN++'s VectorPoolAggregationModule) over stacked
// (ragged) frames: query_stacked_local_neighbor_idxs_wrapper_stack, query_three_nn_by_stacked_local_idxs_wrapper_stack,
// vector_pool_wrapper and vector_pool_grad_wrapper (sm_100a), plus the two kernels of the module's eval path.
//
// Replaces (same lists, dist2 / idx, sums and counts, bit for bit; the order of atomically placed lists and triples is
// free):
//   query_stacked_local_neighbor_idxs_kernel, query_three_nn_by_stacked_local_idxs_kernel, vector_pool_kernel_stack,
//   vector_pool_grad_kernel_stack   (upstream OpenPCDet pointnet2_stack/src/vector_pool_gpu.cu)
//
// Contract (restated from upstream OpenPCDet, not read from this project's reference tree; "recalled" marks what was
// not checked against any source -- the head-to-head tests settle it where the reference is built):
//   * centre p belongs to the first frame k with p < M0 + ... + Mk (stopping at B - 1); its frame's support points are
//     scanned in ascending index; local = support - centre, an fp32 subtract per axis.
//   * neighbor_type 1 (ball): a hit iff fmaf(lz,lz, fmaf(lx,lx, ly*ly)) <= D*D (non-strict; D*D an fp32 product; the
//     contraction is assumed to be the one nvcc chose for the other distance kernels).  Any other type (cube): a hit iff
//     |lx| <= D && |ly| <= D && |lz| <= D.  A NaN coordinate is never a hit here (upstream's `if (d2 > r2) continue`
//     form would take it -- recalled).
//   * local neighbour lists: the first min(hits, 1000 (recalled: temp_idxs[1000]), nsample if > 0) hits as GLOBAL rows;
//     start_len[p] = (atomicAdd(cumsum, L), L); nothing is written at or beyond avg_length * M.
//   * 3-NN over a list: strict-< cascade in list order from sub-voxel centre g, bests (+inf, -1) (the reference's
//     double 1e40 and int -1), so a slot the list cannot fill stays (+inf, -1).  (Some upstream versions may copy slot
//     0 into the unfilled slots -- recalled, not verified.)
//   * vector pool: grid_size_a = D*2 / num_grid_a (fp32), i_a = floorf((l_a + D) / grid_size_a),
//     g = ix*ny*nz + iy*nz + iz clamped as ONE index to [0, G-1] (recalled).  Average pooling, per hit in index order:
//     cnt[p,g] += 1, new_features[p, g*cpg + i % cpg] += f[k,i] for ascending i, new_local_xyz[p, 3g+a] += l_a if
//     use_xyz, one triple (k, p, g), the hit counts toward nsample.  Random choice: only the first hit of each sub-voxel,
//     assigned (=), count 1; stop when (nsample > 0 && taken >= nsample) || taken >= G.  The return value is the exact
//     number of triples a large enough buffer would hold (triples at or beyond num_max_sum_points are not written), so
//     one retry always suffices.
//   * gradient: grad_support[k,i] += grad_new[p, g*cpg + i % cpg] * (1 / max(cnt[p,g], 1)) (atomicAdd; the reciprocal
//     form is recalled).
//
// Design: frame starts come from the stacked ball query's device-side count scan; every frame gets one uniform grid over
// its support points (tsm_grid_build_ragged, cells >= 1.01 D wide, so the 27 cells around a centre hold its ball and its
// cube).  One warp per centre enumerates the hits in ascending index: through the grid, lane l < 27 walks one neighbour
// cell and the warp takes the smallest pending index (the merge walk of the grid ball query), or -- frames whose grid
// is unusable (> 256 points in a cell, a non-finite extent, no points) and TSMDET_BQ_ALGO=brute -- 32 consecutive points
// per step.  Either way the consumer sees one warp-uniform visit per hit, in index order.  The walks are separate from
// the ball query's cores (grid_merge_core, brute_query_core): those write capped index rows with a strict < test, these
// hand every hit's coordinates to a consumer with its own stop rule, and the existing kernels stay byte for byte as they
// were.
//  * lists: the hits are staged in shared memory (<= 1000), then one atomicAdd places the list.
//  * 3-NN (list or fused): the centre's neighbour records are staged in shared memory; lanes own sub-voxels (32 at a
//    time) and run the cascade over the staged records.  The fused form stages the hits of the walk directly: the list
//    is never written and nothing is read back on the host.
//  * vector pool: lanes own output channels, the per-sub-voxel sums live in shared memory and every element is summed in
//    the reference's order; the triples are buffered one per lane and placed 32 at a time.  The planes form writes the
//    eval path's normalised (1, G*(3+C), M) input of the grouped layer instead, and no triples.
//  * interpolation planes: the eval path's (1, G*(C+9), M) input for local_interpolation, straight from the 3-NN.
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "grid.cuh"

namespace tsm {

constexpr int kVpCap = 1000;          // longest neighbour list (the reference's temp_idxs[1000])
constexpr int kVpWarps = 4;           // warps per CTA of the list / 3-NN kernels: 4 x 16 KB of staged records
constexpr int kVpPoolSmem = 200 * 1024;  // shared-memory budget of a vector-pool CTA
constexpr uint32_t kVpNone = 0xffffffffu;

struct VpQuery {
    float cx, cy, cz;
    float d, d2;  // max_neighbour_distance and its fp32 square
    int ball;
};

__device__ __forceinline__ bool vp_hit(float x, float y, float z, const VpQuery& q) {
    const float lx = __fsub_rn(x, q.cx), ly = __fsub_rn(y, q.cy), lz = __fsub_rn(z, q.cz);
    if (q.ball) return __fmaf_rn(lz, lz, __fmaf_rn(lx, lx, __fmul_rn(ly, ly))) <= q.d2;
    return fabsf(lx) <= q.d && fabsf(ly) <= q.d && fabsf(lz) <= q.d;
}

// Every hit of the centre in one frame's grid, ascending frame-local index: one warp-uniform visit(x, y, z, global row)
// per hit until visit returns false.  Lane l < 27 walks neighbour cell (l / 9 - 1, l / 3 % 3 - 1, l % 3 - 1) up to its
// next hit; the warp takes the smallest pending index (redux.sync.min) and its owner moves on.
template <class Visit>
__device__ __forceinline__ void vp_grid_walk(int lane, const GridHdr& h, const int* __restrict__ cell_start,
                                             const float4* __restrict__ sorted, int start, const VpQuery& q,
                                             Visit&& visit) {
    int head = 0, end = 0;
    if (lane < 27) {
        const int gx = grid_q(q.cx, h.lo[0], h.inv[0], h.n[0]) + lane % 3 - 1;
        const int gy = grid_q(q.cy, h.lo[1], h.inv[1], h.n[1]) + (lane / 3) % 3 - 1;
        const int gz = grid_q(q.cz, h.lo[2], h.inv[2], h.n[2]) + lane / 9 - 1;
        if (gx >= 0 && gx < h.n[0] && gy >= 0 && gy < h.n[1] && gz >= 0 && gz < h.n[2]) {
            const int c = (gz * h.n[1] + gy) * h.n[0] + gx;
            head = __ldg(cell_start + c);
            end = __ldg(cell_start + c + 1);
        }
    }
    uint32_t cur = kVpNone;
    float4 rec = make_float4(0.f, 0.f, 0.f, 0.f);
    auto advance = [&]() {
        cur = kVpNone;
        while (head < end) {
            const float4 p = sorted[head];
            ++head;
            if (vp_hit(p.x, p.y, p.z, q)) {
                cur = (uint32_t)__float_as_int(p.w);
                rec = p;
                break;
            }
        }
    };
    advance();
    for (;;) {
        const uint32_t mn = __reduce_min_sync(FULL, cur);
        if (mn == kVpNone) return;
        const int owner = __ffs(__ballot_sync(FULL, cur == mn)) - 1;
        const float x = __shfl_sync(FULL, rec.x, owner), y = __shfl_sync(FULL, rec.y, owner),
                    z = __shfl_sync(FULL, rec.z, owner);
        if (!visit(x, y, z, (int)mn + start)) return;
        if (lane == owner) advance();
    }
}

// The same visits by brute force over the n points (N,3) of one frame: 32 consecutive points per step.
template <class Visit>
__device__ __forceinline__ void vp_brute_walk(int lane, int n, const float* __restrict__ pts, int start, const VpQuery& q,
                                              Visit&& visit) {
    for (int base = 0; base < n; base += 32) {
        const int k = base + lane;
        float x = 0.f, y = 0.f, z = 0.f;
        bool hit = false;
        if (k < n) {
            x = __ldg(pts + 3 * k); y = __ldg(pts + 3 * k + 1); z = __ldg(pts + 3 * k + 2);
            hit = vp_hit(x, y, z, q);
        }
        unsigned bal = __ballot_sync(FULL, hit);
        while (bal) {
            const int j = __ffs(bal) - 1;
            bal &= bal - 1;
            const float hx = __shfl_sync(FULL, x, j), hy = __shfl_sync(FULL, y, j), hz = __shfl_sync(FULL, z, j);
            if (!visit(hx, hy, hz, start + base + j)) return;
        }
    }
}

// The frames' search structures: nstart / mstart (b + 1 exclusive prefix sums), and the grids (hdr == nullptr: none).
struct VpFrames {
    int b;
    const int* nstart;
    const int* mstart;
    const int* hdr;
    const int* cell_start;
    const float4* sorted;
    const float* xyz;
};

template <class Visit>
__device__ __forceinline__ void vp_walk(int lane, const VpFrames& fr, int f, const VpQuery& q, Visit&& visit) {
    const int start = __ldg(fr.nstart + f);
    if (fr.hdr) {
        const GridHdr h = *reinterpret_cast<const GridHdr*>(fr.hdr + (size_t)f * kHdrInts);
        if (h.ok) {
            vp_grid_walk(lane, h, fr.cell_start + (size_t)f * (kGridCells + 1), fr.sorted + start, start, q, visit);
            return;
        }
    }
    vp_brute_walk(lane, __ldg(fr.nstart + f + 1) - start, fr.xyz + (size_t)start * 3, start, q, visit);
}

__device__ __forceinline__ VpQuery vp_query(const float* __restrict__ new_xyz, int p, float d, int ball) {
    VpQuery q;
    q.cx = __ldg(new_xyz + (size_t)p * 3); q.cy = __ldg(new_xyz + (size_t)p * 3 + 1); q.cz = __ldg(new_xyz + (size_t)p * 3 + 2);
    q.d = d;
    q.d2 = __fmul_rn(d, d);
    q.ball = ball;
    return q;
}

// The first `cap` hits of centre p as (x, y, z, global row) records in buf; returns their number (warp-uniform).
__device__ __forceinline__ int vp_stage_hits(int lane, const VpFrames& fr, int p, const VpQuery& q, int cap,
                                             float4* buf) {
    int cnt = 0;
    if (cap > 0)
        vp_walk(lane, fr, stack_frame_of(p, fr.b, fr.mstart), q, [&](float x, float y, float z, int k) {
            if (lane == 0) buf[cnt] = make_float4(x, y, z, __int_as_float(k));
            return ++cnt < cap;
        });
    __syncwarp();
    return cnt;
}

// query_stacked_local_neighbor_idxs: one warp per centre.
__global__ void __launch_bounds__(kVpWarps * 32)
    vp_local_idxs_kernel(int m, VpFrames fr, const float* __restrict__ new_xyz, float d, int ball, int cap,
                         int* __restrict__ stack_idx, int* __restrict__ start_len, int* __restrict__ cumsum,
                         long long max_thresh) {
    extern __shared__ float4 vp_buf[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = blockIdx.x * kVpWarps + warp;
    if (p >= m) return;
    float4* const buf = vp_buf + warp * kVpCap;
    const int cnt = vp_stage_hits(lane, fr, p, vp_query(new_xyz, p, d, ball), cap, buf);
    int off = 0;
    if (lane == 0) {
        off = atomicAdd(cumsum, cnt);
        start_len[2 * (size_t)p] = off;
        start_len[2 * (size_t)p + 1] = cnt;
    }
    off = __shfl_sync(FULL, off, 0);
    for (int j = lane; j < cnt; j += 32)
        if ((long long)off + j < max_thresh) stack_idx[off + j] = __float_as_int(buf[j].w);
}

// The three nearest of the staged records buf[0..len) from (gx, gy, gz): strict-< cascade in record order.
__device__ __forceinline__ void vp_three_nn_scan(const float4* buf, int len, float gx, float gy, float gz, float& b1,
                                                 float& b2, float& b3, int& i1, int& i2, int& i3) {
    for (int j = 0; j < len; ++j) {
        const float4 v = buf[j];
        const float d = sqdist3(v.x, v.y, v.z, gx, gy, gz);
        const int k = __float_as_int(v.w);
        if (d < b1) {
            b3 = b2; i3 = i2;
            b2 = b1; i2 = i1;
            b1 = d; i1 = k;
        } else if (d < b2) {
            b3 = b2; i3 = i2;
            b2 = d; i2 = k;
        } else if (d < b3) {
            b3 = d; i3 = k;
        }
    }
}

// 3-NN of every sub-voxel centre over its centre's neighbours, one warp per centre, lanes over sub-voxels.  FUSED: the
// neighbours are the walk's first `cap` hits (the list query's list, never written); otherwise the list
// stack_idx[start_len[p,0] ...] (length start_len[p,1], clipped to the list_len entries that exist), staged in chunks.
template <bool FUSED>
__global__ void __launch_bounds__(kVpWarps * 32)
    vp_three_nn_kernel(int m, int G, VpFrames fr, const float* __restrict__ new_xyz, float d, int ball, int cap,
                       const int* __restrict__ stack_idx, const int* __restrict__ start_len, long long list_len,
                       int n_total, const float* __restrict__ support_xyz, const float* __restrict__ centres,
                       int* __restrict__ idx, float* __restrict__ dist2) {
    extern __shared__ float4 vp_buf[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p = blockIdx.x * kVpWarps + warp;
    if (p >= m) return;
    float4* const buf = vp_buf + warp * kVpCap;
    int len = 0;
    const int* list = nullptr;
    if (FUSED) {
        len = vp_stage_hits(lane, fr, p, vp_query(new_xyz, p, d, ball), cap, buf);
    } else {
        const long long off = __ldg(start_len + 2 * (size_t)p);
        const long long l = __ldg(start_len + 2 * (size_t)p + 1);
        if (off >= 0 && l > 0 && off < list_len) {
            len = (int)min(l, list_len - off);
            list = stack_idx + off;
        }
    }
    auto stage = [&](int c0, int n) {
        __syncwarp();
        for (int j = lane; j < n; j += 32) {
            const int k = __ldg(list + c0 + j);
            const float nan = __int_as_float(0x7fc00000);  // a row outside the support points is never nearest
            const bool ok = (unsigned)k < (unsigned)n_total;
            buf[j] = make_float4(ok ? __ldg(support_xyz + 3 * (size_t)k) : nan, ok ? __ldg(support_xyz + 3 * (size_t)k + 1) : nan,
                                 ok ? __ldg(support_xyz + 3 * (size_t)k + 2) : nan, __int_as_float(k));
        }
        __syncwarp();
    };
    for (int g0 = 0; g0 < G; g0 += 32) {
        const int g = g0 + lane;
        const size_t r = (size_t)p * G + g;
        float gx = 0.f, gy = 0.f, gz = 0.f;
        if (g < G) { gx = __ldg(centres + 3 * r); gy = __ldg(centres + 3 * r + 1); gz = __ldg(centres + 3 * r + 2); }
        const float inf = __int_as_float(0x7f800000);
        float b1 = inf, b2 = inf, b3 = inf;
        int i1 = -1, i2 = -1, i3 = -1;
        for (int c0 = 0; c0 < len; c0 += kVpCap) {
            const int n = min(kVpCap, len - c0);
            if (!FUSED && (g0 == 0 || len > kVpCap)) stage(c0, n);
            vp_three_nn_scan(buf, n, gx, gy, gz, b1, b2, b3, i1, i2, i3);
        }
        if (g < G) {
            dist2[3 * r] = b1; dist2[3 * r + 1] = b2; dist2[3 * r + 2] = b3;
            idx[3 * r] = i1; idx[3 * r + 1] = i2; idx[3 * r + 2] = i3;
        }
    }
}

struct VpPoolArgs {
    int m, G, ny, nz, cin, cout, cpg, use_xyz, nsample, pooling;
    float d, gsx, gsy, gsz;  // grid_size_a
    int ball;
    const float* new_xyz;
    const float* feats;
    float* new_features;      // (M, cout) rows ...
    float* new_local_xyz;     // (M, 3G)
    int* point_cnt;           // (M, G)
    int* triples;             // (num_max_sum_points, 3)
    int* cum_sum;
    long long max_sum;
    float* planes;            // ... or (1, G*(3+cpg), M) planes
};

// vector_pool: one warp per centre, lanes own output channels (j = lane, lane + 32, ...) of every sub-voxel; the sums
// live in shared memory (per warp: sums[G*cpg], loc[3G], cnt[G]).  PLANES: the CTA's warps take consecutive centres and
// write the normalised planes together once all of them are done.
template <bool PLANES>
__global__ void __launch_bounds__(256, 1) vp_pool_kernel(VpFrames fr, VpPoolArgs a) {
    extern __shared__ float vp_pool_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, W = blockDim.x >> 5;
    const int G = a.G, cpg = a.cpg;
    const int per_warp = G * cpg + 4 * G;
    float* const sums = vp_pool_smem + (size_t)warp * per_warp;
    float* const loc = sums + G * cpg;
    int* const cnt = reinterpret_cast<int*>(loc + 3 * G);
    const int p = blockIdx.x * W + warp;
    if (p < a.m) {
        // the reference adds into (and, random choice, tests) the caller's rows: start from them
        for (int t = lane; t < G * cpg; t += 32)
            sums[t] = PLANES ? 0.f : a.new_features[(size_t)p * a.cout + t];
        for (int t = lane; t < 3 * G; t += 32) loc[t] = PLANES ? 0.f : a.new_local_xyz[(size_t)p * 3 * G + t];
        for (int t = lane; t < G; t += 32) cnt[t] = PLANES ? 0 : a.point_cnt[(size_t)p * G + t];
        __syncwarp();
        const VpQuery q = vp_query(a.new_xyz, p, a.d, a.ball);
        int taken = 0, nbuf = 0, tk = 0, tg = 0;  // lane t holds buffered triple t
        auto flush = [&]() {
            if (PLANES || nbuf == 0) return;
            int base = 0;
            if (lane == 0) base = atomicAdd(a.cum_sum, nbuf);
            base = __shfl_sync(FULL, base, 0);
            if (lane < nbuf && (long long)base + lane < a.max_sum) {
                int* const t = a.triples + 3 * ((size_t)base + lane);
                t[0] = tk; t[1] = p; t[2] = tg;
            }
            nbuf = 0;
        };
        vp_walk(lane, fr, stack_frame_of(p, fr.b, fr.mstart), q, [&](float x, float y, float z, int k) {
            __syncwarp();  // cnt[] written by lane 0 at the previous hit
            const float lx = __fsub_rn(x, q.cx), ly = __fsub_rn(y, q.cy), lz = __fsub_rn(z, q.cz);
            const float mine = lane == 0 ? lx : (lane == 1 ? ly : lz);  // the axis lane a < 3 accumulates
            const int ix = (int)floorf(__fdiv_rn(__fadd_rn(lx, a.d), a.gsx));
            const int iy = (int)floorf(__fdiv_rn(__fadd_rn(ly, a.d), a.gsy));
            const int iz = (int)floorf(__fdiv_rn(__fadd_rn(lz, a.d), a.gsz));
            const int g = min(max(ix * a.ny * a.nz + iy * a.nz + iz, 0), G - 1);
            const float* const f = a.feats + (size_t)k * a.cin;
            if (a.pooling == 0) {
                for (int j = lane; j < cpg; j += 32) {
                    float s = sums[g * cpg + j];
                    for (int i = j; i < a.cin; i += cpg) s = __fadd_rn(s, __ldg(f + i));
                    sums[g * cpg + j] = s;
                }
                if (a.use_xyz && lane < 3) loc[3 * g + lane] = __fadd_rn(loc[3 * g + lane], mine);
                if (lane == 0) cnt[g] += 1;
            } else {
                if (cnt[g] != 0) return true;
                for (int j = lane; j < cpg; j += 32) {
                    float s = 0.f;
                    for (int i = j; i < a.cin; i += cpg) s = __ldg(f + i);  // the last write of the reference's loop
                    if (j < a.cin) sums[g * cpg + j] = s;
                }
                if (a.use_xyz && lane < 3) loc[3 * g + lane] = mine;
                if (lane == 0) cnt[g] = 1;
            }
            if (!PLANES) {
                if (lane == nbuf) { tk = k; tg = g; }
                if (++nbuf == 32) flush();
            }
            ++taken;
            if (a.nsample > 0 && taken >= a.nsample) return false;
            return !(a.pooling != 0 && taken >= G);
        });
        flush();
        __syncwarp();
        if (!PLANES) {
            for (int t = lane; t < G * cpg; t += 32) a.new_features[(size_t)p * a.cout + t] = sums[t];
            if (a.use_xyz)
                for (int t = lane; t < 3 * G; t += 32) a.new_local_xyz[(size_t)p * 3 * G + t] = loc[t];
            for (int t = lane; t < G; t += 32) a.point_cnt[(size_t)p * G + t] = cnt[t];
        }
    }
    if (PLANES) {
        // channel g*(3+cpg) + c: c < 3 the mean local xyz, else the mean feature c - 3; value / max(cnt, 1e-6)
        __syncthreads();
        const int cg = 3 + cpg, nch = G * cg;
        const int p0 = blockIdx.x * W;
        for (int t = threadIdx.x; t < nch * W; t += blockDim.x) {
            const int ch = t / W, w = t - ch * W;
            if (p0 + w >= a.m) continue;
            const float* const ws = vp_pool_smem + (size_t)w * per_warp;
            const int g = ch / cg, c = ch - g * cg;
            const float v = c < 3 ? ws[G * cpg + 3 * g + c] : ws[g * cpg + c - 3];
            const int n = reinterpret_cast<const int*>(ws + G * cpg + 3 * G)[g];
            a.planes[(size_t)ch * a.m + p0 + w] = __fdiv_rn(v, fmaxf((float)n, 1e-6f));
        }
    }
}

// grad_support[k, i] += grad_new[p, g*cpg + i % cpg] * (1 / max(cnt[p,g], 1)) for every triple (k, p, g) and channel i.
__global__ void __launch_bounds__(256)
    vp_pool_grad_kernel(long long work, int n, int m, int G, int cin, int cout, int cpg, const float* __restrict__ grad_new,
                        const int* __restrict__ point_cnt, const int* __restrict__ triples,
                        float* __restrict__ grad_support) {
    for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < work; e += (long long)gridDim.x * 256) {
        const long long t = e / cin;
        const int i = (int)(e - t * cin);
        const int k = __ldg(triples + 3 * t), p = __ldg(triples + 3 * t + 1), g = __ldg(triples + 3 * t + 2);
        if ((unsigned)k >= (unsigned)n || (unsigned)p >= (unsigned)m || (unsigned)g >= (unsigned)G) continue;
        const int c = __ldg(point_cnt + (size_t)p * G + g);
        const float w = __fdiv_rn(1.f, fmaxf((float)c, 1.f));
        atomicAdd(grad_support + (size_t)k * cin + i, __fmul_rn(__ldg(grad_new + (size_t)p * cout + g * cpg + i % cpg), w));
    }
}

// The local_interpolation eval input (1, G*(C+9), M): channel g*(C+9) + c of centre p is, for the sub-voxel row
// r = p*G + g, 0 when idx[r,0] == -1 (no neighbour), else for c < C fmaf(w2,f2, fmaf(w0,f0, w1*f1)) (an index outside
// [0, N) reads 0, as the stacked three_interpolate does) and for c = C + 3s + a centre[r,a] - xyz[idx[r,s], a], a -1 slot
// reading the LAST support row (Python's negative index in the reference module).  32 centres per CTA, written
// through a 32 x 32 shared-memory transpose so that the planes' writes are contiguous.
__global__ void __launch_bounds__(256)
    vp_interp_planes_kernel(int m, int G, int n, int c, const float* __restrict__ features,
                            const float* __restrict__ xyz, const float* __restrict__ centres, const int* __restrict__ idx,
                            const float* __restrict__ weight, float* __restrict__ out) {
    __shared__ float tile[32][33];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int p0 = blockIdx.x * 32;
    const int cg = c + 9;
    const long long nch = (long long)G * cg;
    for (long long c0 = 0; c0 < nch; c0 += 32) {
        const long long ch = c0 + lane;
        const int g = (int)(ch / cg), cc = (int)(ch - (long long)g * cg);
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const int p = p0 + warp + 8 * k;
            float v = 0.f;
            if (p < m && ch < nch) {
                const size_t r = (size_t)p * G + g;
                const int i0 = __ldg(idx + 3 * r);
                if (i0 != -1) {
                    if (cc < c) {
                        float f[3], w[3];
#pragma unroll
                        for (int s = 0; s < 3; ++s) {
                            const int j = s == 0 ? i0 : __ldg(idx + 3 * r + s);
                            w[s] = __ldg(weight + 3 * r + s);
                            f[s] = (unsigned)j < (unsigned)n ? __ldg(features + (size_t)j * c + cc) : 0.f;
                        }
                        v = __fmaf_rn(w[2], f[2], __fmaf_rn(w[0], f[0], __fmul_rn(w[1], f[1])));
                    } else {
                        const int s = (cc - c) / 3, ax = (cc - c) - 3 * s;
                        int j = __ldg(idx + 3 * r + s);
                        if (j < 0) j += n;
                        if ((unsigned)j < (unsigned)n) v = __fsub_rn(__ldg(centres + 3 * r + ax), __ldg(xyz + 3 * (size_t)j + ax));
                    }
                }
            }
            tile[lane][warp + 8 * k] = v;
        }
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const long long cc = c0 + warp + 8 * k;
            const int p = p0 + lane;
            if (cc < nch && p < m) out[(size_t)cc * m + p] = tile[warp + 8 * k][lane];
        }
        __syncthreads();
    }
}

// Frame starts (scratch tag 13) and, unless TSMDET_BQ_ALGO=brute or D is not a usable cell size, the per-frame grids
// over the support points (scratch tag 14).
static int vp_frames(int b, int n_total, float d, const float* xyz, const int* ncnt, const int* mcnt, cudaStream_t stream,
                     VpFrames* fr) {
    void* p = nullptr;
    int rc = tsm_scratch_get(13, sizeof(int) * 2 * ((size_t)b + 1), stream, &p);
    if (rc != TSM_OK) return rc;
    int* const nstart = static_cast<int*>(p);
    int* const mstart = nstart + b + 1;
    rc = tsm_stack_counts_scan(b, ncnt, mcnt, nstart, mstart, stream);
    if (rc != TSM_OK) return rc;
    fr->b = b;
    fr->nstart = nstart;
    fr->mstart = mstart;
    fr->hdr = nullptr;
    fr->cell_start = nullptr;
    fr->sorted = nullptr;
    fr->xyz = xyz;
    const char* algo = tsm_knob(KNOB_BQ_ALGO);
    if (n_total > 0 && d > 0.f && d < 1.0e18f && !(algo && !strcmp(algo, "brute")))
        return tsm_grid_build_ragged(b, n_total, d, nstart, xyz, stream, 14, &fr->hdr, &fr->cell_start, &fr->sorted);
    return TSM_OK;
}

static int vp_cap(int nsample) { return nsample > 0 ? (nsample < kVpCap ? nsample : kVpCap) : kVpCap; }

constexpr int kVpStageSmem = kVpWarps * kVpCap * (int)sizeof(float4);

static int vp_pool_launch(bool planes, int b, int n_total, const float* xyz, const int* ncnt, const int* mcnt,
                          VpPoolArgs& a, cudaStream_t stream) {
    VpFrames fr;
    int rc = vp_frames(b, n_total, a.d, xyz, ncnt, mcnt, stream, &fr);
    if (rc != TSM_OK) return rc;
    const size_t per_warp = sizeof(float) * ((size_t)a.G * a.cpg + 4 * (size_t)a.G);
    if (per_warp > (size_t)kVpPoolSmem) return TSM_ERR_INVALID;
    const int W = (int)(kVpPoolSmem / per_warp < 8 ? kVpPoolSmem / per_warp : 8);
    const int smem = (int)(per_warp * W);
    const unsigned blocks = (unsigned)divup(a.m, W);
    if (planes) {
        TSM_CUDA_TRY(cudaFuncSetAttribute(vp_pool_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        vp_pool_kernel<true><<<blocks, W * 32, smem, stream>>>(fr, a);
    } else {
        TSM_CUDA_TRY(cudaFuncSetAttribute(vp_pool_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        vp_pool_kernel<false><<<blocks, W * 32, smem, stream>>>(fr, a);
    }
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

static bool vp_pool_args(int m, int c_in, int c_out, int ngx, int ngy, int ngz, float d, int use_xyz, int nsample,
                         int neighbor_type, int pooling_type, VpPoolArgs* a) {
    if (ngx <= 0 || ngy <= 0 || ngz <= 0 || c_in < 0 || c_out < 0) return false;
    const long long G = (long long)ngx * ngy * ngz;
    if (G > (1 << 20)) return false;
    memset(a, 0, sizeof(*a));
    a->m = m;
    a->G = (int)G;
    a->ny = ngy;
    a->nz = ngz;
    a->cin = c_in;
    a->cout = c_out;
    a->cpg = (int)(c_out / G);
    a->use_xyz = use_xyz;
    a->nsample = nsample;
    a->pooling = pooling_type;
    a->d = d;
    const float d2 = d * 2.f;  // grid_size_a = max_neighbour_distance * 2 / num_grid_a, fp32
    a->gsx = d2 / (float)ngx;
    a->gsy = d2 / (float)ngy;
    a->gsz = d2 / (float)ngz;
    a->ball = neighbor_type == 1;
    return !(a->cpg == 0 && c_in > 0);
}

}  // namespace tsm

extern "C" {

int tsmdet_stack_local_neighbor_idxs(int b, int m, int n_total, const float* support_xyz, const int* xyz_batch_cnt,
                                     const float* new_xyz, const int* new_xyz_batch_cnt, int* stack_neighbor_idxs,
                                     int* start_len, int* cumsum, int avg_length_of_neighbor_idxs,
                                     float max_neighbour_distance, int nsample, int neighbor_type, void* stream_) {
    using namespace tsm;
    if (m <= 0) return TSM_OK;
    if (b <= 0 || n_total < 0 || !new_xyz || !xyz_batch_cnt || !new_xyz_batch_cnt || !start_len || !cumsum ||
        (n_total > 0 && !support_xyz))
        return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    VpFrames fr;
    int rc = vp_frames(b, n_total, max_neighbour_distance, support_xyz, xyz_batch_cnt, new_xyz_batch_cnt, stream, &fr);
    if (rc != TSM_OK) return rc;
    const long long max_thresh = (long long)avg_length_of_neighbor_idxs * m;
    if (max_thresh > 0 && !stack_neighbor_idxs) return TSM_ERR_INVALID;
    TSM_CUDA_TRY(cudaFuncSetAttribute(vp_local_idxs_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kVpStageSmem));
    vp_local_idxs_kernel<<<(unsigned)divup(m, kVpWarps), kVpWarps * 32, kVpStageSmem, stream>>>(
        m, fr, new_xyz, max_neighbour_distance, neighbor_type == 1, vp_cap(nsample), stack_neighbor_idxs, start_len, cumsum,
        max_thresh);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_stack_three_nn_local(int m, int num_total_grids, int n_total, long long list_len, const float* support_xyz,
                                const float* new_xyz_grid_centers, const int* stack_neighbor_idxs, const int* start_len,
                                int* new_xyz_grid_idxs, float* new_xyz_grid_dist2, void* stream) {
    using namespace tsm;
    if (m <= 0 || num_total_grids <= 0) return TSM_OK;
    if (n_total < 0 || list_len < 0 || !new_xyz_grid_centers || !start_len || !new_xyz_grid_idxs || !new_xyz_grid_dist2 ||
        (list_len > 0 && !stack_neighbor_idxs) || (n_total > 0 && !support_xyz))
        return TSM_ERR_INVALID;
    VpFrames fr = {};
    TSM_CUDA_TRY(cudaFuncSetAttribute(vp_three_nn_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kVpStageSmem));
    vp_three_nn_kernel<false><<<(unsigned)divup(m, kVpWarps), kVpWarps * 32, kVpStageSmem, (cudaStream_t)stream>>>(
        m, num_total_grids, fr, nullptr, 0.f, 0, 0, stack_neighbor_idxs, start_len, list_len, n_total, support_xyz,
        new_xyz_grid_centers, new_xyz_grid_idxs, new_xyz_grid_dist2);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_stack_vector_three_nn(int b, int m, int n_total, int num_total_grids, const float* support_xyz,
                                 const int* xyz_batch_cnt, const float* new_xyz, const int* new_xyz_batch_cnt,
                                 const float* new_xyz_grid_centers, float max_neighbour_distance, int nsample,
                                 int neighbor_type, int* new_xyz_grid_idxs, float* new_xyz_grid_dist2, void* stream_) {
    using namespace tsm;
    if (m <= 0 || num_total_grids <= 0) return TSM_OK;
    if (b <= 0 || n_total < 0 || !new_xyz || !xyz_batch_cnt || !new_xyz_batch_cnt || !new_xyz_grid_centers ||
        !new_xyz_grid_idxs || !new_xyz_grid_dist2 || (n_total > 0 && !support_xyz))
        return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    VpFrames fr;
    int rc = vp_frames(b, n_total, max_neighbour_distance, support_xyz, xyz_batch_cnt, new_xyz_batch_cnt, stream, &fr);
    if (rc != TSM_OK) return rc;
    TSM_CUDA_TRY(cudaFuncSetAttribute(vp_three_nn_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kVpStageSmem));
    vp_three_nn_kernel<true><<<(unsigned)divup(m, kVpWarps), kVpWarps * 32, kVpStageSmem, stream>>>(
        m, num_total_grids, fr, new_xyz, max_neighbour_distance, neighbor_type == 1, vp_cap(nsample), nullptr, nullptr, 0,
        n_total, support_xyz, new_xyz_grid_centers, new_xyz_grid_idxs, new_xyz_grid_dist2);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_stack_vector_pool(int b, int m, int n_total, int c_in, int c_out, const float* support_xyz,
                             const int* xyz_batch_cnt, const float* support_features, const float* new_xyz,
                             const int* new_xyz_batch_cnt, float* new_features, float* new_local_xyz,
                             int* point_cnt_of_grid, int* grouped_idxs, int num_grid_x, int num_grid_y, int num_grid_z,
                             float max_neighbour_distance, int use_xyz, long long num_max_sum_points, int nsample,
                             int neighbor_type, int pooling_type, int* num_cum_sum, float* planes, void* stream_) {
    using namespace tsm;
    VpPoolArgs a;
    if (!vp_pool_args(m, c_in, c_out, num_grid_x, num_grid_y, num_grid_z, max_neighbour_distance, use_xyz, nsample,
                      neighbor_type, pooling_type, &a))
        return TSM_ERR_INVALID;
    cudaStream_t stream = (cudaStream_t)stream_;
    if (!planes) {
        if (!num_cum_sum) return TSM_ERR_INVALID;
        TSM_CUDA_TRY(cudaMemsetAsync(num_cum_sum, 0, sizeof(int), stream));
    }
    if (m <= 0) return TSM_OK;
    if (b <= 0 || n_total < 0 || !new_xyz || !xyz_batch_cnt || !new_xyz_batch_cnt ||
        (n_total > 0 && (!support_xyz || (c_in > 0 && !support_features))) ||
        (!planes && (!new_features || !point_cnt_of_grid || (use_xyz && !new_local_xyz) ||
                     (num_max_sum_points > 0 && !grouped_idxs))))
        return TSM_ERR_INVALID;
    a.new_xyz = new_xyz;
    a.feats = support_features;
    a.new_features = new_features;
    a.new_local_xyz = new_local_xyz;
    a.point_cnt = point_cnt_of_grid;
    a.triples = grouped_idxs;
    a.cum_sum = num_cum_sum;
    a.max_sum = num_max_sum_points;
    a.planes = planes;
    if (planes) a.use_xyz = 1;
    return vp_pool_launch(planes != nullptr, b, n_total, support_xyz, xyz_batch_cnt, new_xyz_batch_cnt, a, stream);
}

int tsmdet_stack_vector_pool_grad(int m, int n, int c_out, int c_in, int num_total_grids, long long num_triples,
                                  const float* grad_new_features, const int* point_cnt_of_grid, const int* grouped_idxs,
                                  float* grad_support_features, void* stream) {
    using namespace tsm;
    if (num_triples <= 0 || c_in <= 0 || n <= 0 || m <= 0) return TSM_OK;
    if (num_total_grids <= 0 || c_out < 0 || !grad_new_features || !point_cnt_of_grid || !grouped_idxs ||
        !grad_support_features)
        return TSM_ERR_INVALID;
    const int cpg = c_out / num_total_grids;
    if (cpg <= 0) return TSM_ERR_INVALID;
    const long long work = num_triples * c_in;
    const long long want = (work + 255) / 256, cap = (long long)tsm_num_sms() * 16;
    vp_pool_grad_kernel<<<(unsigned)(want < cap ? want : cap), 256, 0, (cudaStream_t)stream>>>(
        work, n, m, num_total_grids, c_in, c_out, cpg, grad_new_features, point_cnt_of_grid, grouped_idxs,
        grad_support_features);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

int tsmdet_stack_vector_interp_planes(int m, int num_total_grids, int n, int c, const float* support_features,
                                      const float* support_xyz, const float* new_xyz_grid_centers, const int* idx,
                                      const float* weight, float* planes, void* stream) {
    using namespace tsm;
    if (m <= 0 || num_total_grids <= 0) return TSM_OK;
    if (n < 0 || c < 0 || !new_xyz_grid_centers || !idx || !weight || !planes ||
        (n > 0 && (!support_xyz || (c > 0 && !support_features))))
        return TSM_ERR_INVALID;
    vp_interp_planes_kernel<<<(unsigned)divup(m, 32), 256, 0, (cudaStream_t)stream>>>(
        m, num_total_grids, n, c, support_features, support_xyz, new_xyz_grid_centers, idx, weight, planes);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

}  // extern "C"
