// fps_bucket.cu -- furthest point sampling with exact spatial pruning, one CTA per cloud (N <= 16384).
//
// Replaces (same indices, bit for bit) farthest_point_sampling_kernel / furthest_point_sampling_kernel,
//   /root/reference/pcdet/ops/pointnet2/pointnet2_batch/src/sampling_gpu.cu:100-216, 588-704
// for clouds that fit one SM.  The reference (and fps.cu) touch all N points for every pick: M*N updates.
// A pick only lowers the running min-distance of points closer to it than their current min-distance,
// and after i picks that is ~N/i points.  So:
//
//  * a prologue sorts the cloud into Morton order of an adaptive grid (counting sort in shared memory:
//    histogram -> scan -> scatter), so that every LANE owns P spatially compact points and keeps their
//    bounding box and running min-distances in registers; the coordinates live in shared memory as
//    float4-readable planes (192 KB at N = 16384), the original indices as u16 next to them (32 KB), and
//    one bounding box per 16 lanes in what is left of the 227 KB;
//  * per pick, a lane computes a lower bound of the squared distance from the pick to its group's box with
//    the SAME rounded operations as the point distance (fsub, fmul, 2 fma; each is monotone, so the bound
//    never exceeds any member's computed distance).  If bound >= the lane's largest min-distance no
//    member can change and the lane is skipped; a warp whose 32 lanes all skip does nothing but re-post
//    its cached candidate.  Skipped updates are no-ops by construction, so every min-distance -- and
//    therefore every pick -- is bit-identical to the brute force;
//  * one __syncthreads per pick: warps post (key, position) records, every warp reduces the <= 32
//    records itself (redux.sync), and the reference's tie rule -- among equal maxima the smallest
//    rank(k) = bitrev(k mod bs) : k / bs -- is evaluated lazily, only when a maximum is shared;
//  * K > 1 (clouds of 8193..16384 points): rounds of up to K exact picks decided by a leader warp, with the
//    planes in plain sorted order ("chunk-compact": the 128 points one LDS.128 of a warp reads are spatially
//    compact), one box per half of a warp's chunks, and updates that skip the half a pick cannot reach.
//
// One SM per cloud instead of a cluster of eight, and ~2x fewer cycles per pick: see DESIGN.md 4.1.
#include "fps.cuh"

namespace tsm {
#ifndef FPSB_U1
#define FPSB_U1 4
#endif
constexpr int kU1 = FPSB_U1;
#ifndef FPSB_WAIT
#define FPSB_WAIT 1
#endif
#ifndef FPSB_UPD
#define FPSB_UPD 2
#endif

// -DFPSB_PROF: thread 0 of cloud 0 accumulates clock() per phase of a multi-pick round and prints the totals
#ifdef FPSB_PROF
#define PROF_T(v) const long long v = clock64()
#define PROF_TD(v, dep) const long long v = clock_after((uint32_t)(dep))
__device__ __forceinline__ long long clock_after(uint32_t dep) {  // a clock read that waits for `dep`
    long long t;
    asm volatile("{\n\t.reg .b32 z;\n\tand.b32 z, %1, 0;\n\tcvt.u64.u32 %0, z;\n\t.reg .b64 c;\n\tmov.u64 c, %%clock64;\n\tadd.u64 %0, %0, c;\n\t}" : "=l"(t) : "r"(dep) : "memory");
    return t;
}
#define PROF_ACC(t0, t1, t2, t3)                                                 \
    if (tid == 0) {                                                              \
        prof_apply += t1 - t0; prof_wait += t2 - t1; prof_lead += t3 - t2; ++prof_rounds; \
    }
#define PROF_ACC2(t0, t1, t2, t3, t4, t5)                                        \
    if (tid == 0) {                                                              \
        prof_q[0] += t1 - t0; prof_q[1] += t2 - t1; prof_q[2] += t3 - t2; prof_q[3] += t4 - t3; prof_q[4] += t5 - t4; \
    }
#else
#define PROF_T(v)
#define PROF_TD(v, dep)
#define PROF_ACC(t0, t1, t2, t3)
#define PROF_ACC2(t0, t1, t2, t3, t4, t5)
#endif

constexpr int kBucketMaxN = 16384;
constexpr int kMiscBytes = 512 + 768 + 128 + 16;  // candidate records, box partials, scan offsets, point 0

// planes (12 B per slot) | original indices (2 B per slot) | one box per 16 lanes (24 B); the prologue's cell
// histogram aliases the front
__host__ __device__ __forceinline__ size_t bucket_main_bytes(int cap, int threads, int cell_bits) {
    size_t a = (size_t)14 * cap + (size_t)24 * (threads / 16), h = (size_t)4 << cell_bits;
    size_t mx = a > h ? a : h;
    return (mx + 15) & ~(size_t)15;
}

// sorted position -> shared-memory element index.  A lane owns the elements base + c * 128 + e (chunk c of its warp, e < 4).
// Lane-compact (CH = false): P consecutive sorted points per LANE (a lane's box is tight: the K = 1 loop skips per lane).
// Chunk-compact (CH = true): the planes are simply in sorted order, so chunk c of a warp -- the 128 points ONE LDS.128 of
// the update reads -- is spatially compact and an update can skip whole chunks (multi-pick rounds, see APPLY).
template <int P, bool CH>
__device__ __forceinline__ int slot_index(int s) {
    if (CH) return s;
    const int p = s & (P - 1), l = (s / P) & 31, w = s / (32 * P);
    return w * (32 * P) + (p >> 2) * 128 + l * 4 + (p & 3);
}

__device__ __forceinline__ uint32_t ref_rank(uint32_t k, int L) {
    return (L == 0) ? k : (__brev(k & ((1u << L) - 1u)) | (k >> L));
}

template <int T, int P, int K>
__global__ void __launch_bounds__(T, 1)
    fps_bucket_kernel(const FpsArgs a, const int cell_bits) {
    constexpr int NW = T / 32;
    constexpr int CAP = T * P;
    constexpr int C4 = P / 4;
    constexpr bool CH = K > 1 && C4 >= 2;  // chunk-compact layout, updates skip half of a warp's chunks at a time
    constexpr int HC = CH ? C4 / 2 : C4;   // chunks per half
    extern __shared__ __align__(16) unsigned char dyn[];
    float* const sx = reinterpret_cast<float*>(dyn);
    float* const sy = sx + CAP;
    float* const sz = sy + CAP;
    uint16_t* const sk = reinterpret_cast<uint16_t*>(sz + CAP);         // original index of every slot
    float4* const sbox4 = reinterpret_cast<float4*>(sk + CAP);          // [T/16] {x lo, x hi, y lo, y hi}
    float2* const sbox2 = reinterpret_cast<float2*>(sbox4 + T / 16);    // [T/16] {z lo, z hi}
    uint32_t* const hist = reinterpret_cast<uint32_t*>(dyn);  // prologue only; aliases the planes
    unsigned char* const misc = dyn + bucket_main_bytes(CAP, T, cell_bits);
    uint2* const recs = reinterpret_cast<uint2*>(misc);                      // [2][32] warp candidates
    float* const red = reinterpret_cast<float*>(misc + 512);                 // [6][32] box partials
    uint32_t* const woff = reinterpret_cast<uint32_t*>(misc + 512 + 768);    // [32] scan offsets
    float* const first_xyz = reinterpret_cast<float*>(misc + 512 + 768 + 128);  // point 0

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cloud = blockIdx.x;
    const int n = a.n, m = a.m, L = a.log2bs;
    const float* __restrict__ xyz = a.xyz + (size_t)cloud * n * 3;
    int* __restrict__ idxs = a.idxs + (size_t)cloud * m;
    const bool chain = a.tie_iter != nullptr;

    // ---- chained shortcut (see fps.cu / tsmdet_fps_chain): this cloud is the first n picks of a recorded run
    if (a.parent_tie != nullptr) {
        const bool prefix_ok = a.parent_tie[cloud] >= m && m <= n && n <= a.parent_m &&
                               a.parent_vals[(size_t)cloud * a.parent_m + a.parent_m - 1] > 0.f;
        if (prefix_ok) {
            for (int j = tid; j < m; j += T) {
                idxs[j] = j;
                if (a.vals) a.vals[(size_t)cloud * m + j] = a.parent_vals[(size_t)cloud * a.parent_m + j];
            }
            if (tid == 0 && a.tie_iter) a.tie_iter[cloud] = a.parent_tie[cloud];
            return;
        }
    }
    if (tid == 0 && a.tie_iter) a.tie_iter[cloud] = 0x7fffffff;
    if (tid == 0 && a.vals && m > 0) a.vals[(size_t)cloud * m] = __int_as_float(0x7f800000);

    // ================= prologue: spatial sort =================
    // (1) bounding box of the cloud
    float lo0 = __int_as_float(0x7f800000), lo1 = lo0, lo2 = lo0, hi0 = -lo0, hi1 = -lo0, hi2 = -lo0;
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
        red[0 * 32 + warp] = lo0; red[1 * 32 + warp] = lo1; red[2 * 32 + warp] = lo2;
        red[3 * 32 + warp] = hi0; red[4 * 32 + warp] = hi1; red[5 * 32 + warp] = hi2;
    }
    const int ncells = 1 << cell_bits;
    for (int c = tid; c < ncells; c += T) hist[c] = 0u;
    __syncthreads();
    for (int w = 0; w < NW; ++w) {
        lo0 = fminf(lo0, red[0 * 32 + w]); lo1 = fminf(lo1, red[1 * 32 + w]); lo2 = fminf(lo2, red[2 * 32 + w]);
        hi0 = fmaxf(hi0, red[3 * 32 + w]); hi1 = fmaxf(hi1, red[4 * 32 + w]); hi2 = fmaxf(hi2, red[5 * 32 + w]);
    }
    // (2) grid: cell_bits bits of Morton key, handed out greedily to the axis with the largest cell extent
    float e0 = hi0 - lo0, e1 = hi1 - lo1, e2 = hi2 - lo2;
    if (!(e0 > 0.f) || !(e0 < 3.0e38f)) e0 = 0.f;
    if (!(e1 > 0.f) || !(e1 < 3.0e38f)) e1 = 0.f;
    if (!(e2 > 0.f) || !(e2 < 3.0e38f)) e2 = 0.f;
    int nb0 = 0, nb1 = 0, nb2 = 0;
    uint32_t order = 0u;  // 2 bits per key bit, most significant key bit first
    {
        float c0 = e0, c1 = e1, c2 = e2;
        for (int i = 0; i < cell_bits; ++i) {
            int ax = 0;
            if (c1 > c0 && c1 >= c2) ax = 1;
            if (c2 > c0 && c2 > c1) ax = 2;
            order |= (uint32_t)ax << (2 * i);
            if (ax == 0) { ++nb0; c0 *= 0.5f; }
            else if (ax == 1) { ++nb1; c1 *= 0.5f; }
            else { ++nb2; c2 *= 0.5f; }
        }
    }
    const float inv0 = e0 > 0.f ? (float)(1 << nb0) / e0 : 0.f;
    const float inv1 = e1 > 0.f ? (float)(1 << nb1) / e1 : 0.f;
    const float inv2 = e2 > 0.f ? (float)(1 << nb2) / e2 : 0.f;
    auto cell_key = [&](float x, float y, float z) -> uint32_t {
        const int q0 = min(max(__float2int_rd((x - lo0) * inv0), 0), (1 << nb0) - 1);
        const int q1 = min(max(__float2int_rd((y - lo1) * inv1), 0), (1 << nb1) - 1);
        const int q2 = min(max(__float2int_rd((z - lo2) * inv2), 0), (1 << nb2) - 1);
        int r0 = nb0, r1 = nb1, r2 = nb2;
        uint32_t key = 0u;
        for (int i = 0; i < cell_bits; ++i) {
            const uint32_t ax = (order >> (2 * i)) & 3u;
            uint32_t bit;
            if (ax == 0u) bit = (q0 >> --r0) & 1;
            else if (ax == 1u) bit = (q1 >> --r1) & 1;
            else bit = (q2 >> --r2) & 1;
            key = (key << 1) | bit;
        }
        return key;
    };
    // (3) histogram over cells; this thread's points are k = tid + i*T (coalesced reads)
    uint32_t packed[P / 2];  // two u16 per register: first the cell keys, later the sorted positions
#pragma unroll
    for (int i = 0; i < P; ++i) {
        const int k = tid + i * T;
        uint32_t key = 0xffffu;
        if (k < n) {
            key = cell_key(__ldg(xyz + 3 * k), __ldg(xyz + 3 * k + 1), __ldg(xyz + 3 * k + 2));
            atomicAdd(&hist[key], 1u);
        }
        if (i & 1) packed[i >> 1] |= key << 16;
        else packed[i >> 1] = key;
    }
    __syncthreads();
    // (4) exclusive scan of the histogram: warp w owns ncells/NW consecutive cells
    {
        const int cpw = ncells / NW;
        uint32_t carry = 0u;
        for (int c = warp * cpw + lane; c < (warp + 1) * cpw; c += 32) {
            const uint32_t v = hist[c];
            uint32_t inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += t;
            }
            hist[c] = carry + inc - v;
            carry += __shfl_sync(FULL, inc, 31);
        }
        if (lane == 0) woff[warp] = carry;
        __syncthreads();
        if (warp == 0) {
            const uint32_t v = lane < NW ? woff[lane] : 0u;
            uint32_t inc = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(FULL, inc, o);
                if (lane >= o) inc += t;
            }
            if (lane < NW) woff[lane] = inc - v;
        }
        __syncthreads();
        // (5) sorted position of every point (order inside a cell is arbitrary -- it only decides which lane
        //     owns a point, never a result)
        const int cshift = cell_bits - (31 - __clz(NW));  // log2(cpw)
#pragma unroll
        for (int i = 0; i < P; ++i) {
            const uint32_t key = (i & 1) ? (packed[i >> 1] >> 16) : (packed[i >> 1] & 0xffffu);
            uint32_t s = 0xffffu;
            if (key != 0xffffu) s = atomicAdd(&hist[key], 1u) + woff[key >> cshift];
            if (i & 1) packed[i >> 1] = (packed[i >> 1] & 0xffffu) | (s << 16);
            else packed[i >> 1] = (packed[i >> 1] & 0xffff0000u) | s;
        }
    }
    __syncthreads();  // the histogram is dead; its bytes become the coordinate planes
    // (6) scatter coordinates + original index to the sorted position; zero the padding slots
    for (int s = n + tid; s < CAP; s += T) {
        const int e = slot_index<P, CH>(s);
        sx[e] = 0.f; sy[e] = 0.f; sz[e] = 0.f; sk[e] = 0;
    }
#pragma unroll
    for (int i = 0; i < P; ++i) {
        const int k = tid + i * T;
        if (k < n) {
            const uint32_t s = (i & 1) ? (packed[i >> 1] >> 16) : (packed[i >> 1] & 0xffffu);
            const int e = slot_index<P, CH>((int)s);
            sx[e] = __ldg(xyz + 3 * k);
            sy[e] = __ldg(xyz + 3 * k + 1);
            sz[e] = __ldg(xyz + 3 * k + 2);
            sk[e] = (uint16_t)k;
        }
    }
    __syncthreads();

    // ================= per-lane state =================
    const int base = warp * (32 * P) + lane * 4;    // element index of this lane's slot 0
    const int first = (warp * 32 + lane) * P;       // sorted position of slot 0 (lane-compact layout)
    auto slot_valid = [&](int p) -> bool {          // slot p of this lane holds a point of the cloud
        return CH ? (base + (p >> 2) * 128 + (p & 3) < n) : (first + p < n);
    };
    float md[P];
    {
        // Order each lane's P points by ascending reference rank (any order inside a lane is as good as another
        // for the pruning), so that "lowest slot among equal maxima" IS the reference's tie rule inside a lane.
        // Slots past the cloud's end take the largest ranks and stay last.  Chunk-compact layout: the order is established
        // inside every group of 4 slots only (a point must stay in its chunk); equal maxima in different chunks of one lane
        // -- different points at equal distances, rare -- are decided by an explicit rank comparison in warp_argmax.
        uint32_t rk[P];
#pragma unroll
        for (int p = 0; p < P; ++p)
            rk[p] = slot_valid(p) ? ref_rank(sk[base + (p >> 2) * 128 + (p & 3)], L) : (0xffffffe0u + (uint32_t)p);
        int dst[P];  // element index each slot's point moves to
#pragma unroll
        for (int p = 0; p < P; ++p) {
            int before = CH ? (p & ~3) : 0;
#pragma unroll
            for (int q = 0; q < P; ++q)
                if (!CH || (q >> 2) == (p >> 2)) before += (rk[q] < rk[p]) ? 1 : 0;
            dst[p] = base + (before >> 2) * 128 + (before & 3);
        }
        {
            uint16_t v[P];
#pragma unroll
            for (int p = 0; p < P; ++p) v[p] = sk[base + (p >> 2) * 128 + (p & 3)];
#pragma unroll
            for (int p = 0; p < P; ++p) sk[dst[p]] = v[p];
        }
#pragma unroll
        for (int pl = 0; pl < 3; ++pl) {
            float* const plane = sx + pl * CAP;
            float v[P];
#pragma unroll
            for (int p = 0; p < P; ++p) v[p] = plane[base + (p >> 2) * 128 + (p & 3)];
#pragma unroll
            for (int p = 0; p < P; ++p) plane[dst[p]] = v[p];
        }
        // (only this thread touches these elements: no barrier needed before it reads them back)
    }
#pragma unroll
    for (int h = 0; h < (CH ? 2 : 1); ++h) {
        float bx0 = __int_as_float(0x7f800000), by0 = bx0, bz0 = bx0, bx1 = -bx0, by1 = -bx0, bz1 = -bx0;
#pragma unroll
        for (int c = h * HC; c < (h + 1) * HC; ++c) {
            const float4 X = *reinterpret_cast<const float4*>(sx + base + c * 128);
            const float4 Y = *reinterpret_cast<const float4*>(sy + base + c * 128);
            const float4 Z = *reinterpret_cast<const float4*>(sz + base + c * 128);
            const float xs[4] = {X.x, X.y, X.z, X.w}, ys[4] = {Y.x, Y.y, Y.z, Y.w}, zs[4] = {Z.x, Z.y, Z.z, Z.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
                const int p = c * 4 + e;
                float d0 = -2.f;
                if (slot_valid(p)) {
                    bx0 = fminf(bx0, xs[e]); bx1 = fmaxf(bx1, xs[e]);
                    by0 = fminf(by0, ys[e]); by1 = fmaxf(by1, ys[e]);
                    bz0 = fminf(bz0, zs[e]); bz1 = fmaxf(bz1, zs[e]);
                    d0 = a.temp ? a.temp[(size_t)cloud * n + sk[base + c * 128 + e]] : 1e10f;
                }
                md[p] = d0;
            }
        }
        // one box per 16 lanes (what fits next to the planes): union over the half-warp; chunk-compact layout: one box
        // per half of the warp's chunks (box 2 * warp + h), union over the warp
#pragma unroll
        for (int o = CH ? 16 : 8; o > 0; o >>= 1) {
            bx0 = fminf(bx0, __shfl_xor_sync(FULL, bx0, o)); bx1 = fmaxf(bx1, __shfl_xor_sync(FULL, bx1, o));
            by0 = fminf(by0, __shfl_xor_sync(FULL, by0, o)); by1 = fmaxf(by1, __shfl_xor_sync(FULL, by1, o));
            bz0 = fminf(bz0, __shfl_xor_sync(FULL, bz0, o)); bz1 = fmaxf(bz1, __shfl_xor_sync(FULL, bz1, o));
        }
        if (CH ? lane == 0 : (lane & 15) == 0) {
            const int bi = CH ? 2 * warp + h : tid >> 4;
            sbox4[bi] = make_float4(bx0, bx1, by0, by1);
            sbox2[bi] = make_float2(bz0, bz1);
        }
    }
    if (tid == 0) {
        idxs[0] = 0;
        first_xyz[0] = __ldg(xyz + 0);
        first_xyz[1] = __ldg(xyz + 1);
        first_xyz[2] = __ldg(xyz + 2);
    }
    __syncthreads();

    // lane state: (lmax, u, lpos) = this lane's largest min-distance and where it is; warp state (wu, wpos) = the
    // warp's candidate, wu2 = an upper bound (as a key) of every OTHER point of the warp
    float lmax = -2.f;
    uint32_t u = 0u, wu = 0u, wpos = (uint32_t)base, wu2 = 0u;
    int lpos = base;

    // lower bound of the computed squared distance from a pick to the lane's box, with the point formula's own
    // rounded operations
    auto box_bound = [&](float x1, float y1, float z1, const float4 b4, const float2 b2) -> float {
        const float dx = fmaxf(fmaxf(__fsub_rn(b4.x, x1), __fsub_rn(x1, b4.y)), 0.f);
        const float dy = fmaxf(fmaxf(__fsub_rn(b4.z, y1), __fsub_rn(y1, b4.w)), 0.f);
        const float dz = fmaxf(fmaxf(__fsub_rn(b2.x, z1), __fsub_rn(z1, b2.y)), 0.f);
        return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
    };
    // chunks [q0, q1) of this lane (all of them by default)
    auto update = [&](float x1, float y1, float z1, const int q0, const int q1) {  // (constants at every call site)
        const unsigned long long nx = f2_pack(-x1, -x1), ny = f2_pack(-y1, -y1), nz = f2_pack(-z1, -z1);
#pragma unroll
        for (int q = 0; q < C4; ++q) {
            if (q < q0 || q >= q1) continue;
            const float4 X = *reinterpret_cast<const float4*>(sx + base + q * 128);
            const float4 Y = *reinterpret_cast<const float4*>(sy + base + q * 128);
            const float4 Z = *reinterpret_cast<const float4*>(sz + base + q * 128);
            const float2 d01 = sqdist3_x2(nx, ny, nz, X.x, X.y, Y.x, Y.y, Z.x, Z.y);  // FADD2 / FMUL2 / FFMA2: bit-identical
            const float2 d23 = sqdist3_x2(nx, ny, nz, X.z, X.w, Y.z, Y.w, Z.z, Z.w);  // to sqdist3, half the instructions
            md[q * 4 + 0] = fminf(d01.x, md[q * 4 + 0]);
            md[q * 4 + 1] = fminf(d01.y, md[q * 4 + 1]);
            md[q * 4 + 2] = fminf(d23.x, md[q * 4 + 2]);
            md[q * 4 + 3] = fminf(d23.y, md[q * 4 + 3]);
        }
    };
    // The lane / warp argmax after an update.  Leaves (wu, wpos, wu2); bit 31 of wpos = "another point of this warp
    // with different coordinates shares wu" (chain bookkeeping).
    auto warp_argmax = [&]() {
        // balanced max tree over the P slots; for K > 1 it also carries the runner-up (which equals the maximum when
        // the maximum is held twice: min(a, b) of two equal maxima)
        float t[P], t2[P];
#pragma unroll
        for (int p = 0; p < P; ++p) { t[p] = md[p]; t2[p] = -2.f; }
#pragma unroll
        for (int w = 1; w < P; w <<= 1) {
#pragma unroll
            for (int p = 0; p + w < P; p += 2 * w) {
                if (K > 1) t2[p] = fmaxf(fminf(t[p], t[p + w]), fmaxf(t2[p], t2[p + w]));
                t[p] = fmaxf(t[p], t[p + w]);
            }
        }
        lmax = t[0];
        u = (lmax > -1.f) ? f32_ordered(lmax) : 0u;  // the reference starts from best = -1
        // where this lane's maximum sits: the lowest slot among equals (slots are in reference-rank order)
        uint32_t eq = 0u;
#pragma unroll
        for (int p = 0; p < P; ++p) eq |= (md[p] == lmax) ? (1u << p) : 0u;
        int bp = __ffs(eq) - 1;
        const bool several = (eq & (eq - 1u)) != 0u;
        if (CH && several && (eq & ~((2u << (bp | 3)) - 1u)) != 0u) {
            // (rare) the maximum sits in several chunks of this lane: slots are in rank order inside a chunk only, so the
            // lowest maximum of every chunk competes by reference rank
            uint32_t rest = eq, brk = 0xffffffffu;
            while (rest) {
                const int p = __ffs(rest) - 1;
                rest &= ~(0xfu << (p & ~3));
                const uint32_t r = ref_rank(sk[base + (p >> 2) * 128 + (p & 3)], L);
                if (r < brk) { brk = r; bp = p; }
            }
        }
        lpos = base + (bp >> 2) * 128 + (bp & 3);
        // the warp's candidate: one redux, one ballot, one shuffle (bit 31: the lane holds several maxima)
        wu = __reduce_max_sync(FULL, u);
        const unsigned tie = __ballot_sync(FULL, u == wu);
        wpos = __shfl_sync(FULL, (uint32_t)lpos | (several ? 0x80000000u : 0u), __ffs(tie) - 1);
        const bool lane_tie = (wpos >> 31) != 0u;
        wpos &= 0x7fffffffu;
        if (K > 1) {
            // the runner-up key: the largest in the warp once the candidate itself is set aside (a second lane or slot
            // holding the maximum makes it equal to wu)
            const uint32_t u2 = (t2[0] > -1.f) ? f32_ordered(t2[0]) : 0u;
            wu2 = __reduce_max_sync(FULL, (lane == __ffs(tie) - 1) ? u2 : u);
        }
        if (wu != 0u && ((tie & (tie - 1u)) != 0u || ((chain || K > 1) && lane_tie))) {
            // shared maximum inside the warp: the reference rank decides between lanes, and bit 31 of the candidate
            // says whether a point with DIFFERENT coordinates shares it (chain bookkeeping; runner-up below)
            const uint32_t rk = (u == wu) ? ref_rank(sk[lpos], L) : 0xffffffffu;
            const uint32_t wrk = __reduce_min_sync(FULL, rk);
            const int wl = __ffs(__ballot_sync(FULL, rk == wrk)) - 1;
            wpos = (uint32_t)__shfl_sync(FULL, lpos, wl);
            if (chain || K > 1) {
                bool other = false;
                if (u == wu) {
                    const float fx = sx[wpos], fy = sy[wpos], fz = sz[wpos];
                    uint32_t rest = eq;
                    while (rest) {
                        const int p = __ffs(rest) - 1;
                        rest &= rest - 1u;
                        const int e = base + (p >> 2) * 128 + (p & 3);
                        other |= sx[e] != fx || sy[e] != fy || sz[e] != fz;
                    }
                }
                other = __any_sync(FULL, other);
                if (chain && other) wpos |= 0x80000000u;
                if (K > 1 && !other) {
                    // every point sharing the maximum is an exact duplicate of the candidate: picking the candidate
                    // zeroes them, so the runner-up that matters is the largest key among the OTHER points
                    float s2 = -2.f;
#pragma unroll
                    for (int p = 0; p < P; ++p) s2 = fmaxf(s2, (u == wu && md[p] == lmax) ? -2.f : md[p]);
                    wu2 = __reduce_max_sync(FULL, (s2 > -1.f) ? f32_ordered(s2) : 0u);
                }
            }
        }
    };
    // The pick among the posted records (held one per lane): largest key, smallest reference rank among equals.
    // Returns the record lane; `other` = chain bookkeeping (a different point shares the maximum).
    auto first_pick = [&](const uint2 r, const uint32_t gu, const unsigned gt, uint32_t& cpos, bool& other) -> int {
        int gl = __ffs(gt) - 1;
        cpos = __shfl_sync(FULL, r.y, gl);
        other = (cpos >> 31) != 0u;
        if ((gt & (gt - 1u)) != 0u) {  // several warps share the maximum
            const uint32_t rk = (r.x == gu) ? ref_rank(sk[r.y & 0x7fffffffu], L) : 0xffffffffu;
            const uint32_t grk = __reduce_min_sync(FULL, rk);
            gl = __ffs(__ballot_sync(FULL, rk == grk)) - 1;
            cpos = __shfl_sync(FULL, r.y, gl);
            if (chain) {
                const int e = (int)(r.y & 0x7fffffffu), w = (int)(cpos & 0x7fffffffu);
                other = __any_sync(FULL, r.x == gu && ((r.y >> 31) != 0u || sx[e] != sx[w] || sy[e] != sy[w] ||
                                                      sz[e] != sz[w]));
            }
        }
        return gl;
    };

    float4 b4 = sbox4[tid >> 4];
    float2 b2 = sbox2[tid >> 4];
    if constexpr (K == 1) {
        // ================= one barrier per pick =================
        // Every warp posts its (cached or refreshed) candidate, then reduces the NW records itself.
        float x1 = first_xyz[0], y1 = first_xyz[1], z1 = first_xyz[2];
        for (int j = 1; j < m; ++j) {
            uint2* const rec = recs + (j & 1) * 32;  // double-buffered: a fast warp may already post pick j+1
            const bool hit = !(box_bound(x1, y1, z1, b4, b2) >= lmax) || j == 1;  // NaN bounds count as hits
            if (__any_sync(FULL, hit)) {
                update(x1, y1, z1, 0, C4);
                warp_argmax();
            }
            if (lane == 0) rec[warp] = make_uint2(wu, wpos);
            __syncthreads();
            uint2 r = make_uint2(0u, 0u);
            if (lane < NW) r = rec[lane];
            // the group's box lives in shared memory (registers are short during the update); fetched here, in the
            // shadow of the reduction, for the next pick's test
            b4 = sbox4[tid >> 4];
            b2 = sbox2[tid >> 4];
            const uint32_t gu = __reduce_max_sync(FULL, r.x);
            const unsigned gt = __ballot_sync(FULL, r.x == gu);
            if (gu == 0u) {  // no eligible candidate anywhere: the reference yields index 0
                x1 = first_xyz[0];
                y1 = first_xyz[1];
                z1 = first_xyz[2];
                if (tid == 0) {
                    idxs[j] = -1;
                    if (a.vals) a.vals[(size_t)cloud * m + j] = 0.f;
                }
                continue;
            }
            uint32_t cpos;
            bool other;
            first_pick(r, gu, gt, cpos, other);
            const int gpos = (int)(cpos & 0x7fffffffu);
            x1 = sx[gpos];
            y1 = sy[gpos];
            z1 = sz[gpos];
            if (tid == ((j & (NW - 1)) << 5)) {  // bookkeeping rotates over the warps
                // the slot for now (fire-and-forget store); translated to the original index after the loop
                idxs[j] = gpos;
                if (a.vals) a.vals[(size_t)cloud * m + j] = __uint_as_float(gu & 0x7fffffffu);
                if (chain && other) atomicMin(a.tie_iter + cloud, j);
            }
        }
    } else {
        // ================= rounds of up to K picks =================
        // Measured on B200 with clock64(): warp collectives (SHFL / VOTE / REDUX) cost ~30-50 cycles each and do not
        // overlap inside one warp; a lone warp issues dependent instructions ~4.5 cycles apart; and every instruction an
        // idle warp issues is taken from the few warps with real work.  So a round is organised around shared memory:
        //  * APPLY: a warp reads its hit masks over the round's picks (three words, one per helper).  Zero -> it does
        //    nothing.  Otherwise the P updates run for the picks that may reach it, and it re-runs its argmax and posts
        //    (key, position, runner-up key, sort key) only if its candidate point itself was lowered.
        //  * DECIDE (leader = warp 0, lane w = warp w's record): every lane finds its record's sorted position by
        //    comparing its sort key against all 32 (8 LDS.128); position k < K is adopted by lane k through a
        //    position table; the K (K-1) / 2 "does pick i lower candidate k" tests run one pair per lane; one ballot
        //    yields the number of picks.  Position 0 is the plain argmax (largest key, smallest reference rank among
        //    equals; records within 32 ulp of the top are re-examined exactly).  The candidate q at position k is ALSO
        //    the pick that would follow -- with no update in between -- when
        //      (i)   no other warp's candidate has a key within 32 ulp of q's (the order needs no rank decision),
        //      (ii)  its key is strictly larger than the runner-up key of every warp an earlier pick of this round came
        //            from (exact duplicates of that warp's candidate excepted: picking the candidate zeroes them), and
        //      (iii) no earlier pick of this round changes it: !(sqdist(pick, q) < md[q]), the update's own expression;
        //    every other point is below q now and updates only lower min-distances, so q is the exact next argmax.  The
        //    round stops at the first position that fails a test.
        //  * HELPERS (warps 1..3, one per other SM sub-partition) meanwhile test each candidate against every warp's two
        //    group boxes and current maximum: the hit masks of the next APPLY.
        // Barriers: 1 = "records posted" (bar.arrive by everyone, bar.sync by the leader), 3 = "candidates written"
        // (leader arrives, helpers wait), 2 = "round decided" (everyone).
        uint32_t* const rkey = reinterpret_cast<uint32_t*>(misc);          // [32] warp candidates: key
        uint32_t* const rpos = rkey + 32;                                  // [32] position (bit 31: chain bookkeeping)
        uint32_t* const rkey2 = rkey + 64;                                 // [32] runner-up key
        uint32_t* const rskey = rkey + 96;                                 // [32] sort key: (key & ~31) | (31 - warp), unique
        uint32_t* const posarr = rkey + 128;                               // [32] leader: sorted position of a record
        uint32_t* const sk_at = rkey + 160;                                // [32] leader: sort key at a position
        uint32_t* const whitp = rkey + 192;                                // [3][32] per helper, per warp: picks that may reach it
        float4* const cand = reinterpret_cast<float4*>(rkey + 288);        // [K] the round's candidates / picks: x, y, z
        uint32_t* const ckey = rkey + 320;                                 // [K] ... their keys
        uint32_t* const cr2 = rkey + 328;                                  // [K] ... the runner-up keys of their warps
        int* const npick = reinterpret_cast<int*>(rkey + 336);             // how many of them are picks
        static_assert(K <= 8 && NW >= 4 && 338 * 4 <= 512 + 768 + 128, "round state must fit the prologue scratch");
        constexpr int kBarPost = 1, kBarDone = 2, kBarCand = 3;
        __syncthreads();  // the prologue scratch is dead
        if (tid < 32) {
            rkey[tid] = 0u;
            rpos[tid] = 0u;
            rkey2[tid] = 0u;
            rskey[tid] = 31u - tid;
            posarr[tid] = 0x7fu;
            sk_at[tid] = 0u;
            whitp[tid] = CH ? 0x0101u : 1u;  // round 0: every warp applies pick 0 (to both halves of its chunks)
            whitp[32 + tid] = 0u;
            whitp[64 + tid] = 0u;
        }
        if (tid < K) cand[tid] = make_float4(first_xyz[0], first_xyz[1], first_xyz[2], 0.f);
        if (tid == 0) *npick = 1;
        int c = 1;  // picks of the round being applied
        __syncthreads();
#ifdef FPSB_PROF
        long long prof_apply = 0, prof_wait = 0, prof_lead = 0, prof_rounds = 0, prof_t00 = clock64();
        long long prof_q[5] = {0, 0, 0, 0, 0};
        long long pw_hits = 0, pw_rounds = 0, pw_redo = 0, pw_upd = 0, pw_arg = 0, pw_c = 0, pw_u1 = 0;  // per warp: APPLY phase
#endif
        int round = 0;
        for (int j = 1; j < m; ++round) {
            PROF_T(tp0);
            // ---- APPLY the round's picks (cand[0..c)); j = the first pick the leader decides next
            // (no second, finer test here: the round is bound by the latency of this chain, not by issue slots, so an
            // update that turns out to change nothing is cheaper than a test + warp vote that might avoid it)
            // chunk-compact layout: bits 0..7 = picks that may reach the first half of the warp's chunks, 8..15 = the second
            const unsigned wm2 = (whitp[warp] | whitp[32 + warp] | whitp[64 + warp]) & (((1u << c) - 1u) * (CH ? 0x0101u : 1u));
            const unsigned wm = CH ? ((wm2 | (wm2 >> 8)) & 0xffu) : wm2;
#ifdef FPSB_PROF
            const long long pw0 = clock_after(wm);
            long long pw1 = pw0;
#endif
            if (wm != 0u) {
                // The warp's record stays valid as long as its candidate point itself is not lowered: updates only lower
                // min-distances, so the maximum stays where it is and the runner-up key stays an upper bound.  The test
                // is the update's own expression on the candidate, evaluated by every lane alike (no vote).
                const float cx = sx[wpos & 0x7fffffffu], cy = sy[wpos & 0x7fffffffu], cz = sz[wpos & 0x7fffffffu];
                const float cval = __uint_as_float(wu & 0x7fffffffu);
                // no valid record yet (first round, ineligible warp), or a hit record that says a point with different
                // coordinates shares its maximum: that point may just have been lowered, and a stale bit would record a
                // tie the one-pick algorithm never sees (tie_iter too early, chained shortcut lost)
                bool redo = (wu & 0x80000000u) == 0u || (wpos >> 31) != 0u;
#ifdef FPSB_PROF
                const long long pwc = clock_after(__float_as_uint(cx) ^ __float_as_uint(cy) ^ __float_as_uint(cz));
                pw_c += pwc - pw0;
#endif
                // (only the bit positions first..last set: a lone warp pays ~5 cycles per instruction, and scanning all K
                //  positions cost more than the ~1.2 updates a hit warp applies per round)
#pragma unroll 1
                for (int k = __ffs(wm) - 1; (wm >> k) != 0u; ++k) {
                    if ((wm >> k) & 1u) {
                        const float4 pk = cand[k];
                        redo |= sqdist3(pk.x, pk.y, pk.z, cx, cy, cz) < cval;
#ifdef FPSB_PROF
                        const long long pu0 = clock_after(__float_as_uint(pk.x) ^ __float_as_uint(pk.z));
#endif
                        if (CH) {  // warp-uniform: whole LDS.128 / FADD2 ... groups are skipped, not lanes
                            if ((wm2 >> k) & 1u) update(pk.x, pk.y, pk.z, 0, HC);
                            if ((wm2 >> (k + 8)) & 1u) update(pk.x, pk.y, pk.z, HC, C4);
                        } else {
                            update(pk.x, pk.y, pk.z, 0, C4);
                        }
#ifdef FPSB_PROF
                        uint32_t dep = 0u;
#pragma unroll
                        for (int p = 0; p < P; ++p) dep ^= __float_as_uint(md[p]);
                        pw_u1 += clock_after(dep) - pu0;
#endif
                    }
                }
#ifdef FPSB_PROF
                pw1 = clock_after(__float_as_uint(md[0]) ^ __float_as_uint(md[P - 1]));
                pw_hits += __popc(wm); ++pw_rounds; pw_redo += redo ? 1 : 0;
#endif
                if (redo) {
                    warp_argmax();
                    if (lane == 0) {
                        rkey[warp] = wu;
                        rpos[warp] = wpos;
                        rkey2[warp] = wu2;
                        rskey[warp] = (wu & ~31u) | (31u - (uint32_t)warp);
                    }
                }
#ifdef FPSB_PROF
                const long long pw2 = clock_after(wu ^ wu2);
                pw_upd += pw1 - pw0; pw_arg += pw2 - pw1;
#endif
            }
            if (warp != 0) {
                asm volatile("bar.arrive %0, %1;" ::"n"(kBarPost), "n"(T) : "memory");
                if (warp < 4) {
                    // ---- HELPER h = warp - 1: which of the candidates h, h+3, ... may reach warp `lane`?  A candidate
                    // reaches a warp when the bound to one of its two group boxes is below the warp's current maximum.
                    asm volatile("bar.sync %0, 128;" ::"n"(kBarCand) : "memory");
                    const uint32_t wkey = rkey[lane];
                    const float wmax = (wkey & 0x80000000u) ? __uint_as_float(wkey & 0x7fffffffu)
                                                            : (wkey == 0u ? -__int_as_float(0x7f800000) : __int_as_float(0x7f800000));
                    const int g = 2 * (lane & (NW - 1));
                    const float4 g0 = sbox4[g], g1 = sbox4[g + 1];
                    const float2 h0 = sbox2[g], h1 = sbox2[g + 1];
                    unsigned hmask = 0u;
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        if (k % 3 != warp - 1) continue;
                        const float4 ck = cand[k];
                        const bool hit0 = !(box_bound(ck.x, ck.y, ck.z, g0, h0) >= wmax), hit1 = !(box_bound(ck.x, ck.y, ck.z, g1, h1) >= wmax);
                        if (CH) hmask |= (hit0 ? (1u << k) : 0u) | (hit1 ? (0x100u << k) : 0u);
                        else hmask |= (hit0 || hit1) ? (1u << k) : 0u;
                    }
                    whitp[32 * (warp - 1) + lane] = hmask;
                }
            } else {
                PROF_T(tp1);
                asm volatile("bar.sync %0, %1;" ::"n"(kBarPost), "n"(T) : "memory");
                PROF_T(tp2);
                // ---- DECIDE picks j, j+1, ...
                const uint32_t mykey = rkey[lane];
                PROF_TD(tq0, mykey);
                // Sorted position of every record.  The sort key drops the 5 lowest bits of the key and carries the warp
                // instead, so keys are unique and one compare per record places a record; records whose keys agree in
                // the upper 27 bits ("near ties", incl. real ties) are ordered arbitrarily and are re-examined below.
                const uint32_t mysk = rskey[lane];
                int pos;
                {
                    int gt[2] = {0, 0};
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const uint4 k4 = reinterpret_cast<const uint4*>(rskey)[q];
                        gt[q & 1] += (k4.x > mysk ? 1 : 0) + (k4.y > mysk ? 1 : 0) + (k4.z > mysk ? 1 : 0) + (k4.w > mysk ? 1 : 0);
                    }
                    pos = gt[0] + gt[1];
                }
                PROF_TD(tq1, pos);
                posarr[lane] = (uint32_t)pos;
                if (pos <= K && mykey != 0u) sk_at[pos] = mysk;
                __syncwarp();
                // lane k < K adopts the record at position k (a stale table entry fails the position check)
                const uint32_t skk = sk_at[lane & 15], skn = sk_at[(lane & 15) + 1], skp = sk_at[(lane + 15) & 15];
                uint32_t src = 31u - (skk & 31u);
                bool valid = lane < K && posarr[src] == (uint32_t)lane && rkey[src] != 0u;
                const bool near_tie = (skk >> 5) == (skn >> 5) || (lane != 0 && (skk >> 5) == (skp >> 5));
                bool shared_key = false;
                if (lane == 0 && valid && near_tie) {
                    // (rare) the plain argmax among the records near the top: largest key, smallest reference rank
                    uint32_t bk = 0u, brk = 0xffffffffu;
                    for (int l = 0; l < NW; ++l) {
                        if ((rskey[l] >> 5) != (skk >> 5)) continue;
                        const uint32_t kl = rkey[l];
                        if (kl < bk) continue;
                        const uint32_t rl = ref_rank(sk[rpos[l] & 0x7fffffffu], L);
                        if (kl > bk) {
                            bk = kl; brk = rl; src = (uint32_t)l; shared_key = false;
                        } else {
                            shared_key = true;
                            if (rl < brk) { brk = rl; src = (uint32_t)l; }
                        }
                    }
                }
                const uint32_t qkey = rkey[src], qr2 = rkey2[src];
                uint32_t qpos = rpos[src];
                const int qe = (int)(qpos & 0x7fffffffu);
                float qx = sx[qe], qy = sy[qe], qz = sz[qe];
                if (lane == 0 && !valid) {  // no eligible candidate anywhere: the reference yields index 0
                    qx = first_xyz[0];
                    qy = first_xyz[1];
                    qz = first_xyz[2];
                }
                PROF_TD(tq2, __float_as_uint(qx) ^ __float_as_uint(qy) ^ __float_as_uint(qz) ^ qr2);
                if (lane < K) {
                    cand[lane] = make_float4(qx, qy, qz, 0.f);
                    ckey[lane] = qkey;
                    cr2[lane] = qr2;
                }
                __syncwarp();
                asm volatile("bar.arrive %0, 128;" ::"n"(kBarCand) : "memory");  // the helpers may start
                const float qmd = __uint_as_float(qkey & 0x7fffffffu);  // the record's min-distance (keys of values >= 0)
                // test (iii), one (earlier, later) pair of positions per lane: does the earlier one change the later one?
                bool pmoved = false;
                {
                    int hi = 1;  // pair index `lane` -> positions lo < hi: pairs of hi start at hi (hi - 1) / 2
#pragma unroll
                    for (int t = 2; t < K; ++t) hi += (lane >= t * (t - 1) / 2) ? 1 : 0;
                    const int lo = lane - hi * (hi - 1) / 2;
                    if (lane < K * (K - 1) / 2) {
                        const float4 pl = cand[lo], ph = cand[hi];
                        pmoved = sqdist3(pl.x, pl.y, pl.z, ph.x, ph.y, ph.z) < __uint_as_float(ckey[hi] & 0x7fffffffu);
                    }
                }
                const unsigned pm = __ballot_sync(FULL, pmoved);
                const bool moved = lane < K && ((pm >> (lane * (lane - 1) / 2)) & ((1u << lane) - 1u)) != 0u;
                // test (ii): the runner-up keys of the earlier positions' warps
                uint32_t run2 = 0u;
#pragma unroll
                for (int q = 0; q < (K + 3) / 4; ++q) {
                    const uint4 v = reinterpret_cast<const uint4*>(cr2)[q];
                    run2 = max(run2, 4 * q + 0 < lane ? v.x : 0u);
                    run2 = max(run2, 4 * q + 1 < lane ? v.y : 0u);
                    run2 = max(run2, 4 * q + 2 < lane ? v.z : 0u);
                    run2 = max(run2, 4 * q + 3 < lane ? v.w : 0u);
                }
                // keys of positive finite values lie in (0x80000000, 0xff800000); anything else ends the round
                // (and a later record whose maximum a point with different coordinates shares: an earlier pick of the
                // round may lower that point, after which the one-pick algorithm records no tie)
                const bool ok = lane == 0 || (valid && !near_tie && j + lane < m && qkey > run2 && qkey > 0x80000000u &&
                                              qkey < 0xff800000u && !moved && (qpos >> 31) == 0u);
                PROF_TD(tq3, (ok ? 1u : 0u));
                const unsigned okm = __ballot_sync(FULL, ok);
                const int cnt = __ffs(~okm) - 1;  // the leading run of accepted positions
                PROF_TD(tq4, cnt);
                PROF_ACC2(tp2, tq0, tq1, tq2, tq3, tq4);
                if (lane < cnt) {
                    bool other = (qpos >> 31) != 0u;  // chain bookkeeping: a different point shares the maximum
                    float val = qmd;
                    if (lane == 0) {
                        *npick = cnt;
                        if (!valid) {
                            qpos = 0xffffffffu;
                            val = 0.f;
                            other = false;
                        } else if (chain && shared_key) {
                            for (int l = 0; l < NW; ++l) {
                                if (rkey[l] != qkey) continue;
                                const uint32_t e2 = rpos[l];
                                const int e = (int)(e2 & 0x7fffffffu);
                                other |= (e2 >> 31) != 0u || sx[e] != qx || sy[e] != qy || sz[e] != qz;
                            }
                        }
                    }
                    // the slot for now (fire-and-forget store); translated to the original index after the loop
                    idxs[j + lane] = (qpos == 0xffffffffu) ? -1 : (int)(qpos & 0x7fffffffu);
                    if (a.vals) a.vals[(size_t)cloud * m + j + lane] = val;
                    if (chain && other) atomicMin(a.tie_iter + cloud, j + lane);
                }
                PROF_T(tp3);
                PROF_ACC(tp0, tp1, tp2, tp3);
            }
            asm volatile("bar.sync %0, %1;" ::"n"(kBarDone), "n"(T) : "memory");
            c = *npick;
            j += c;
        }
        if (a.temp != nullptr && c > 1) {
            // temp leaves with the min-distances to picks 0..m-2 (the reference never applies its last pick): the last
            // round's picks but the final one are still outstanding
            const unsigned wm2 = (whitp[warp] | whitp[32 + warp] | whitp[64 + warp]) & (((1u << (c - 1)) - 1u) * (CH ? 0x0101u : 1u));
#pragma unroll 1
            for (int k = 0; k < K; ++k) {
                const float4 pk = cand[k];
                if ((wm2 >> k) & 1u) update(pk.x, pk.y, pk.z, 0, HC);
                if (CH && ((wm2 >> (k + 8)) & 1u)) update(pk.x, pk.y, pk.z, HC, C4);
            }
        }
#ifdef FPSB_PROF
        if (lane == 0 && cloud == 0)
            printf("   warp %2d: hit in %lld rounds, %lld updates, %lld argmax;  cycles per hit round: one update %lld; cand coords %lld, updates (incl.) %lld, argmax+post %lld\n", warp,
                   pw_rounds, pw_hits, pw_redo, pw_u1 / (pw_hits ? pw_hits : 1), pw_c / (pw_rounds ? pw_rounds : 1), pw_upd / (pw_rounds ? pw_rounds : 1), pw_arg / (pw_rounds ? pw_rounds : 1));
        if (tid == 0 && cloud == 0)
            printf("fpsb K=%d n=%d m=%d rounds %lld  cycles/round: apply(warp0) %lld  wait-for-posts %lld  leader %lld  total %lld\n",
                   K, n, m, prof_rounds, prof_apply / prof_rounds, prof_wait / prof_rounds, prof_lead / prof_rounds,
                   (clock64() - prof_t00) / prof_rounds);
        if (tid == 0 && cloud == 0)
            printf("   leader: barrier wait %lld  positions %lld  adopt %lld  tests %lld  ballot %lld\n", prof_q[0] / prof_rounds,
                   prof_q[1] / prof_rounds, prof_q[2] / prof_rounds, prof_q[3] / prof_rounds, prof_q[4] / prof_rounds);
#endif
    }

    __syncthreads();  // every idxs[j] slot store of this CTA is visible to it
    for (int j = 1 + tid; j < m; j += T) {
        const int e = idxs[j];
        idxs[j] = e >= 0 ? (int)sk[e] : 0;
    }
    if (a.temp) {
#pragma unroll
        for (int p = 0; p < P; ++p) {
            if (slot_valid(p)) a.temp[(size_t)cloud * n + sk[base + (p >> 2) * 128 + (p & 3)]] = md[p];
        }
    }
}

template <int T, int P, int K>
static int launch_bucket(const FpsArgs& a, int b, int cell_bits, cudaStream_t stream) {
    auto kern = fps_bucket_kernel<T, P, K>;
    const size_t dyn = bucket_main_bytes(T * P, T, cell_bits) + kMiscBytes;
    if (dyn > 227 * 1024) return TSM_ERR_INVALID;
    if (dyn > 40 * 1024) TSM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)dyn));
    kern<<<b, T, dyn, stream>>>(a, cell_bits);
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}

// one pick per barrier (K = 1), or rounds of up to 4 picks where the CTA has the helper warps for it
template <int T, int P>
static int launch_bucket_k(const FpsArgs& a, int b, int cell_bits, cudaStream_t stream, int K) {
    if constexpr (T >= 128) {
        if (K > 1) return launch_bucket<T, P, 4>(a, b, cell_bits, stream);
    }
    return launch_bucket<T, P, 1>(a, b, cell_bits, stream);
}

}  // namespace tsm

bool tsm_fps_bucket_supports(int n, bool weighted) { return !weighted && n >= 1 && n <= tsm::kBucketMaxN; }

// Launch shape: T threads x P points per lane >= n.  Measured on B200 (profiles/r01_fps_bucket_sweep.txt): 8
// points per lane up to 1024 threads, then more points per lane -- 1024 x 16 at N = 16384 (0.67 us per pick,
// 512 x 32: 0.70).  Overridable with TSMDET_FPSB_T / TSMDET_FPSB_P.
int tsm_fps_bucket_launch(const tsm::FpsArgs& a, int b, cudaStream_t stream) {
    const int n = a.n;
    if (!tsm_fps_bucket_supports(n, a.weights != nullptr)) return TSM_ERR_INVALID;
    int T = 0, P = 0;
    if (const char* e = tsm_knob(KNOB_FPSB_T)) T = atoi(e);
    if (const char* e = tsm_knob(KNOB_FPSB_P)) P = atoi(e);
    if (P != 4 && P != 8 && P != 16 && P != 32) P = 0;
    if (T != 32 && T != 64 && T != 128 && T != 256 && T != 512 && T != 1024) T = 0;
    if (T && P && (long)T * P < n) T = P = 0;
    if (T && !P) {
        for (int p = 4; p <= 32 && !P; p <<= 1)
            if ((long)T * p >= n) P = p;
        if (!P) T = 0;
    }
    if (!T) {
        if (!P) P = 8;
        T = 32;
        while (T < 1024 && (long)T * P < n) T <<= 1;
        while ((long)T * P < n && P < 32) P <<= 1;
    }
    if ((long)T * P > tsm::kBucketMaxN || P > 32) return TSM_ERR_INVALID;
    int lg = 0;
    while ((1 << lg) < n) ++lg;
    int cell_bits = lg + 1;
    if (cell_bits < 10) cell_bits = 10;
    if (cell_bits > 15) cell_bits = 15;
    // Picks per round (see the kernel).  Measured on B200 (profiles/r01_fps_multipick.txt): rounds of up to 8 picks pay
    // for clouds of 8193..16384 points (1024 x 16: 2.74 -> 1.80 ms at 16384 -> 4096, 2.04 ms on duplicate-padded
    // clouds); smaller clouds keep one pick per barrier.  TSMDET_FPSB_K = 1 | 2 | 4 | 8 overrides.
    int K = (T == 1024 && P == 16) ? 8 : 1;
    if (const char* e = tsm_knob(KNOB_FPSB_K)) K = atoi(e);
#define FPSB_CASE(TT, PP)                                                               \
    if (T == TT && P == PP) return tsm::launch_bucket_k<TT, PP>(a, b, cell_bits, stream, K);
#define FPSB_CASE_K(TT, PP)                                                             \
    if (T == TT && P == PP && K == 2) return tsm::launch_bucket<TT, PP, 2>(a, b, cell_bits, stream); \
    if (T == TT && P == PP && K == 8) return tsm::launch_bucket<TT, PP, 8>(a, b, cell_bits, stream);
    FPSB_CASE_K(1024, 16)
#ifndef FPSB_QUICK  // (development: compile one launch shape only)
    FPSB_CASE_K(512, 8) FPSB_CASE_K(128, 8)
    FPSB_CASE(32, 4) FPSB_CASE(64, 4) FPSB_CASE(128, 4) FPSB_CASE(256, 4) FPSB_CASE(512, 4) FPSB_CASE(1024, 4)
    FPSB_CASE(32, 8) FPSB_CASE(64, 8) FPSB_CASE(128, 8) FPSB_CASE(256, 8) FPSB_CASE(512, 8) FPSB_CASE(1024, 8)
    FPSB_CASE(32, 16) FPSB_CASE(64, 16) FPSB_CASE(128, 16) FPSB_CASE(256, 16) FPSB_CASE(512, 16) FPSB_CASE(1024, 16)
    FPSB_CASE(32, 32) FPSB_CASE(64, 32) FPSB_CASE(128, 32) FPSB_CASE(256, 32) FPSB_CASE(512, 32)
#else
    FPSB_CASE(1024, 16)
#endif
#undef FPSB_CASE_K
#undef FPSB_CASE
    return TSM_ERR_INVALID;
}
