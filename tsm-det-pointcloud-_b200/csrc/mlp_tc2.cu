// mlp_tc2.cu -- second-generation tcgen05 shared-MLP kernel: the fused set-abstraction scale (gather -> mask ->
// [1x1 conv + ReLU]* -> max over nsample; /root/reference/pcdet/ops/pointnet2/pointnet2_batch/pointnet2_modules.py:
// 1259-1268, 1297-1300) and the point-wise MLPs of the same file (PointnetFPModule.mlp :175-176, aggregation_mlp
// :1320-1321: [1x1 conv + ReLU]* over a dense (B,C,n) tensor, no pooling) in one template.
//
// What changed against sa_mlp_tc.cu (kept for nsample < 8 and as the A/B reference, TSMDET_MLP_V1=1), and why:
//
//  * THE LAST LAYER IS COMPUTED TRANSPOSED.  Both operands are K-major core-matrix images in shared memory, so the
//    roles can be swapped for free: D^T[channel, row] = W_last (A operand, M = 128 output channels per block) x
//    activations (B operand, N = the tile's 128 rows).  In TMEM a lane is now an output CHANNEL and the columns are the
//    tile's rows, i.e. the nsample rows of a centre are consecutive columns of ONE thread: the max-pool is an
//    in-register FMNMX3 tree (16 instructions per 32 samples) instead of one REDUX.SYNC per channel per warp, and bias +
//    ReLU run once per centre AFTER the pool (both are monotone, so max(relu(x+b)) == relu(max(x)+b) bit for bit).  The
//    dense mode uses the same layout to write 256 contiguous bytes per thread.
//  * THE BIAS OF EVERY OTHER LAYER IS ADDED BY THE TENSOR CORE: one extra K step multiplies a constant "ones" operand
//    ([1, 1, 0, ...] per row, part of the weight image) with two weight rows holding bf16(b) and bf16(b - bf16(b)); the
//    sum reproduces the fp32 bias to 2^-17 relative.  The mid-layer epilogue is then tcgen05.ld -> F2FP.RELU -> STS: no
//    shared-memory bias loads and no adds (a third of its instructions in the round-2 ncu source view).
//  * TWO THREADS PER TILE ROW (256-thread tile groups): ncu of the one-thread-per-row version showed 8 warps per SM at
//    23 % issue slots, each warp a ~1800-instruction dependent chain per tile (28 % of the samples on the MMA barrier,
//    the rest latency of its own chain).  Now thread (row, h) drains column half h in the epilogues and gathers the
//    chunks of parity h: half the chain per warp, twice the warps.  Epilogue widths are compile-time (switch over the
//    usual layer widths) and the pooling epilogue has a check-free path for whole tiles.
//  * epilogues keep two 32-column tcgen05.ld in flight per wait::ld and convert with F2FP.RELU (ReLU for free);
//  * rows are gathered a whole tile ahead into registers (or as cp.async, LDGSTS with zero-fill for masked rows, for
//    rows wider than 128 channels); the neighbour indices are prefetched one tile further ahead; one group barrier per
//    layer;
//  * kernel parameters are __grid_constant__ (the per-layer plan arrays are indexed dynamically: without it the
//    compiler copies them to local memory).
//
// One CTA = GROUPS x 256 threads; a group = one independent 128-row tile pipeline (own operand buffer, TMEM
// columns, mbarrier, named barrier) over the CTA's resident weights, persistent over tiles.
#include <cstdio>
#include <cstring>
#include <type_traits>

#include "sa_mlp.cuh"
#include "umma.cuh"

// -DMLP_PROF: lane 0 of warp 1 (a non-issuing warp) of group 0 of CTA 0 accumulates clock64() per phase of a tile and
// prints the per-tile averages when the kernel ends (TSMDET_NVCC_EXTRA=-DMLP_PROF python .../build.py --force)
#ifdef MLP_PROF
#define MPROF(i)                                                        \
    do {                                                                \
        if (prof_on) {                                                  \
            const long long t_ = clock64();                             \
            prof_acc[i] += t_ - prof_t;                                 \
            prof_t = t_;                                                \
        }                                                               \
    } while (0)
#else
#define MPROF(i)
#endif

namespace tsm {

constexpr int T2_ROWS = 128;
constexpr int T2_MAX_LAYERS = 4;

struct Tc2Plan {
    int nl;
    int eb;                    // bytes per operand element: 2 = bf16 (kind::f16), 4 = tf32 (kind::tf32)
    int cl;                    // CTAs per tile: 1, or 2 = a cluster pair, each CTA holding HALF of every layer's output channels
    int K[T2_MAX_LAYERS];      // padded input channels of layer l (multiple of a K step: 16 bf16 / 8 tf32), without the bias step
    int Npad[T2_MAX_LAYERS];   // rows of layer l's weight image IN ONE CTA: cout padded to 16 (last layer: to 128), / cl
    int w_off[T2_MAX_LAYERS];  // byte offset of layer l's weights (non-last layers: K + 16 input rows, the last 16 = bias step)
    int b_off;                 // byte offset of the LAST layer's bias (fp32; added after the pool)
    int ones_off;              // the bias step's A operand: 2 chunk planes x 128 rows, [1, 1, 0, ...] | zeros
    int a_off, a_bytes;        // activation operand buffers (one per tile group)
    int x_off;                 // nsample == 128: per-group exchange of the two halves' maxima (2 x 128 floats), else -1
    int smem_bytes, packed_bytes;  // packed_bytes: one CTA's image (the whole image is cl of them, rank-major)
    int cp;                    // SA mode: feature channels padded to 8 (width of the bf16 transpose)
    int xyz_chunk;             // SA mode: 16-byte chunk index of [dx,dy,dz,0...] in layer-0 rows, -1 if unused
    int grp_cols, tmem_cols;   // TMEM columns of one tile group / of the CTA (power of two >= 32)
    int mb;                    // 128-channel blocks of the (transposed) last layer
    int whole_tiles;           // SA mode: M % (centres per tile) == 0 -> a tile's centres share the frame, consecutive p
    int cls_off;               // SA mode, width-class tiles: the tile table + per-group centre ids in shared memory, else -1
    int ncls;                  // width classes: log2(nsample) + 1
};

// ---- Width-class tiles (SA mode).  A centre is computed on the first w = 2^k rows of its nsample (w <= nsample) when
// every idx slot j >= w repeats one of slots 0 .. w-1: then the dropped rows are byte copies of kept rows (same
// neighbour, same centre, same mask), and
//  * each output element of a tcgen05.mma depends only on its own A row and the weights (the bitwise tests against
//    TSMDET_MLP_WIDTH=fixed confirm this on the hardware), so a copied row yields the same activations through
//    every layer -- the mid-layer biases are per row, the last layer's bias and ReLU come after the pool;
//  * the max over a set is unchanged by dropping duplicates.
// So the width-class path is bit-identical to the fixed-width one.  sa_width_classify_kernel takes the smaller of two
// widths it can prove from the row itself: next_pow2(cnt) when slots cnt.. are the cyclic padding the batch ball query
// writes (row[j] == row[j mod cnt]: every value lies in slots 0 .. cnt-1), and next_pow2(t) when slots t.. all repeat
// slot 0 (padding with the first hit, and hand-made rows).  A row that fits neither keeps nsample; an empty ball (cnt
// <= 0: every row zeroed) has width 1.  It writes, per class k, the centre ids of that class into region k of a list
// (order within a class is arbitrary; empty balls as ~id), and the class sizes; a class-k tile holds 128 >> k centres,
// w rows each, the last tile of a class may be partial.  Tiles run class by class; the table of tile ranges is built by
// every CTA from the class sizes, on the device, so the step needs no host synchronisation.
constexpr int T2_MAX_CLS = 8;     // nsample <= 128
constexpr int T2_CLS_LIST = 32;   // ints before the lists: the class sizes
__global__ void __launch_bounds__(256) sa_width_classify_kernel(const int* __restrict__ idx, const int* __restrict__ cnt,
                                                                const int centres, const int ns, int* __restrict__ cls) {
    __shared__ int s_n[T2_MAX_CLS], s_base[T2_MAX_CLS];
    if (threadIdx.x < T2_MAX_CLS) s_n[threadIdx.x] = 0;
    __syncthreads();
    const int i = blockIdx.x * 256 + threadIdx.x;
    int k = -1, v = 0;
    if (i < centres) {
        const int* r = idx + (size_t)i * ns;
        const int c = cnt != nullptr ? min(__ldg(cnt + i), ns) : ns;
        const int i0 = __ldg(r);
        int t = 1;         // 1 + the last slot that differs from slot 0
        bool cyc = c > 0;  // slots c.. are row[j mod c]
        for (int j = 1; j < ns; ++j) {
            const int x = __ldg(r + j);
            if (x != i0) t = j + 1;
            if (j >= c && cyc && x != __ldg(r + j % c)) cyc = false;
        }
        if (cyc && c < t) t = c;
        const bool empty = c <= 0;
        if (empty) t = 1;
        k = 32 - __clz(t - 1);  // ceil(log2(t))
        v = empty ? ~i : i;
    }
    const unsigned peers = __match_any_sync(FULL, k);
    const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
    int wb = 0;
    if (k >= 0 && lane == leader) wb = atomicAdd(&s_n[k], __popc(peers));
    wb = __shfl_sync(FULL, wb, leader) + __popc(peers & ((1u << lane) - 1u));
    __syncthreads();
    if (threadIdx.x < T2_MAX_CLS && s_n[threadIdx.x] > 0) s_base[threadIdx.x] = atomicAdd(cls + threadIdx.x, s_n[threadIdx.x]);
    __syncthreads();
    if (k >= 0) cls[T2_CLS_LIST + (size_t)k * centres + s_base[k] + wb] = v;
}

// Weights (cout,cin) fp32 + bias -> the kernel's shared-memory image: per layer bf16 [K/8 (+2)][Npad][8] (UMMA K-major
// core matrices; non-last layers end with the two planes of the bias step: input row K = bf16(b), row K+1 = bf16(b -
// bf16(b)), rows K+2.. = 0), the last layer's fp32 bias, the ones operand.  SA mode: layer 0's input channels are
// permuted to the operand order [features 0..C-1 | pad to cp | dx,dy,dz | pad] (reference order: [dx,dy,dz,
// features...], pointnet2_utils.py:523).  blockIdx.y == nl builds the ones operand and the last bias.
__global__ void __launch_bounds__(256) pack_weights2_kernel(const SaMlpArgs a, const Tc2Plan pl, const int dense,
                                                            unsigned char* __restrict__ packed) {
    const int l = blockIdx.y;
    const int rank = blockIdx.z;  // cluster pair: CTA `rank` holds output channels [rank * Npad, (rank + 1) * Npad) of every layer
    packed += (size_t)rank * pl.packed_bytes;
    const int epc = 16 / pl.eb, ks = 2 * epc;  // elements per 16-byte chunk, per K step
    auto put = [&](unsigned char* base, size_t e, float v) {
        if (pl.eb == 2) reinterpret_cast<__nv_bfloat16*>(base)[e] = __float2bfloat16_rn(v);
        else reinterpret_cast<uint32_t*>(base)[e] = to_tf32(v);
    };
    auto rnd = [&](float v) { return pl.eb == 2 ? __bfloat162float(__float2bfloat16_rn(v)) : __uint_as_float(to_tf32(v)); };
    if (l == pl.nl) {
        for (int e = blockIdx.x * 256 + threadIdx.x; e < 2 * T2_ROWS * epc; e += gridDim.x * 256)
            put(packed + pl.ones_off, e, (e < T2_ROWS * epc && (e % epc) < 2) ? 1.f : 0.f);
        const int Np = pl.Npad[pl.nl - 1], cout = a.ch[pl.nl];
        float* bs = reinterpret_cast<float*>(packed + pl.b_off);
        for (int e = blockIdx.x * 256 + threadIdx.x; e < Np; e += gridDim.x * 256)
            bs[e] = rank * Np + e < cout ? __ldg(a.bias[pl.nl - 1] + rank * Np + e) : 0.f;
        return;
    }
    const int K = pl.K[l], Np = pl.Npad[l];
    const int Kb = K + (l + 1 < pl.nl ? ks : 0);  // + the bias step
    const int cin = a.ch[l], cout = a.ch[l + 1];
    const float* __restrict__ W = a.w[l];
    for (int e = blockIdx.x * 256 + threadIdx.x; e < Np * Kb; e += gridDim.x * 256) {
        const int k = e / Np, n = e - k * Np;  // consecutive threads -> consecutive n: 16-byte-strided writes
        const int ng = rank * Np + n;          // the output channel
        float o = 0.f;
        if (ng < cout) {
            if (k >= K) {
                const float b = __ldg(a.bias[l] + ng);
                if (k == K) o = rnd(b);
                else if (k == K + 1) o = b - rnd(b);
            } else {
                int src = -1;
                if (l == 0 && !dense) {
                    if (k < a.c_feat)
                        src = (a.use_xyz ? 3 : 0) + k;
                    else if (pl.xyz_chunk >= 0 && k >= pl.xyz_chunk * epc && k < pl.xyz_chunk * epc + 3)
                        src = k - pl.xyz_chunk * epc;
                } else if (k < cin) {
                    src = k;
                }
                if (src >= 0) o = __ldg(W + (size_t)ng * cin + src);
            }
        }
        put(packed + pl.w_off[l], (size_t)(k / epc) * (Np * epc) + n * epc + (k % epc), o);
    }
}

// features (B,C,N) fp32 -> (B,N,Cp) bf16, zero padded to Cp channels.  One CTA moves a 64-point x Cp-channel tile
// through shared memory: the reads run along N (coalesced 256-byte rows of one channel), the writes along Cp (the 64
// output rows of the tile are ONE contiguous run of 64 * Cp bf16) -- the first version wrote 16-byte pieces 2*Cp bytes
// apart and needed 14 us for the 8 MB of SA layer 3; HBM-bound it is ~2 us.
constexpr int TR_PTS = 64;
template <typename OutT>  // __nv_bfloat16, or float holding tf32-rounded values
__global__ void __launch_bounds__(256) transpose2_kernel(int c, int cp, int n, const float* __restrict__ f, OutT* __restrict__ out) {
    extern __shared__ __align__(16) unsigned char tr_raw[];
    OutT* const tr_tile = reinterpret_cast<OutT*>(tr_raw);  // [TR_PTS][ld] (odd word stride: conflict-free column writes)
    const int b = blockIdx.y;
    const int i0 = blockIdx.x * TR_PTS;
    const int np = min(TR_PTS, n - i0);
    const int ld = cp + (sizeof(OutT) == 2 ? 2 : 1);
    const float* src = f + (size_t)b * c * n + i0;
    for (int e = threadIdx.x; e < cp * TR_PTS; e += 256) {
        const int ch = e / TR_PTS, p = e - ch * TR_PTS;
        float v = 0.f;
        if (ch < c && p < np) v = __ldg(src + (size_t)ch * n + p);
        if constexpr (sizeof(OutT) == 2) tr_tile[p * ld + ch] = __float2bfloat16_rn(v);
        else tr_tile[p * ld + ch] = __uint_as_float(to_tf32(v));
    }
    __syncthreads();
    // 4-byte stores, consecutive threads -> consecutive words of the contiguous output run
    uint32_t* dst = reinterpret_cast<uint32_t*>(out + ((size_t)b * n + i0) * cp);
    constexpr int EPW = 4 / (int)sizeof(OutT);  // elements per word
    const int wpr = cp / EPW;                   // words per output row
    for (int e = threadIdx.x; e < np * wpr; e += 256) {
        const int p = e / wpr, w = e - p * wpr;
        dst[e] = *reinterpret_cast<const uint32_t*>(tr_tile + p * ld + EPW * w);
    }
}

// ReLU + operand-type pack of NC accumulator columns of this thread's row -> 16-byte chunks of the next layer's A
// operand (8 bf16 or 4 tf32 per chunk).  (The bias is already in the accumulator: every non-last layer ends with one
// extra K step against the constant "ones" operand whose weight rows hold bias_hi + bias_lo, so the epilogue has no
// shared-memory bias loads and no adds.)
// REMOTE: the chunk also goes to the same place in the peer CTA's operand buffer (rdst = its shared::cluster address).
__device__ __forceinline__ void st_cluster_v4(uint32_t raddr, const uint4 v) {
    asm volatile("st.shared::cluster.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(raddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int NC, int EB, bool REMOTE>
__device__ __forceinline__ void epi_mid_store(const uint32_t (&v)[NC], unsigned char* dst, uint32_t rdst) {
    if constexpr (EB == 2) {
#pragma unroll
        for (int q = 0; q < NC / 8; ++q) {
            const uint4 o = make_uint4(
                pack_bf16_relu(__uint_as_float(v[8 * q + 0]), __uint_as_float(v[8 * q + 1])),
                pack_bf16_relu(__uint_as_float(v[8 * q + 2]), __uint_as_float(v[8 * q + 3])),
                pack_bf16_relu(__uint_as_float(v[8 * q + 4]), __uint_as_float(v[8 * q + 5])),
                pack_bf16_relu(__uint_as_float(v[8 * q + 6]), __uint_as_float(v[8 * q + 7])));
            *reinterpret_cast<uint4*>(dst + (size_t)q * (T2_ROWS * 16)) = o;
            if constexpr (REMOTE) st_cluster_v4(rdst + (uint32_t)q * (T2_ROWS * 16), o);
        }
    } else {
#pragma unroll
        for (int q = 0; q < NC / 4; ++q) {
            const uint4 o =
                make_uint4(to_tf32(fmaxf(__uint_as_float(v[4 * q + 0]), 0.f)), to_tf32(fmaxf(__uint_as_float(v[4 * q + 1]), 0.f)),
                           to_tf32(fmaxf(__uint_as_float(v[4 * q + 2]), 0.f)), to_tf32(fmaxf(__uint_as_float(v[4 * q + 3]), 0.f)));
            *reinterpret_cast<uint4*>(dst + (size_t)q * (T2_ROWS * 16)) = o;
            if constexpr (REMOTE) st_cluster_v4(rdst + (uint32_t)q * (T2_ROWS * 16), o);
        }
    }
}

// HW accumulator columns starting at TMEM address `taddr` (this thread's lane) -> chunk planes starting at dst;
// compile-time width: straight-line code, two 32-column loads in flight per wait where the width allows
template <int HW, bool LEAN, int EB, bool REMOTE>
__device__ __forceinline__ void epi_mid(uint32_t taddr, unsigned char* dst, uint32_t rdst) {
    constexpr int EPC = 16 / EB;  // columns per chunk plane
    constexpr uint32_t PL = T2_ROWS * 16;
    if constexpr (LEAN && HW >= 64) {  // 128-register kernels: one 32-column load in flight
#pragma unroll
        for (int i = 0; i < HW / 32; ++i)
            epi_mid<32, false, EB, REMOTE>(taddr + 32u * i, dst + (size_t)(32 * i / EPC) * PL, rdst + (uint32_t)(32 * i / EPC) * PL);
        return;
    }
    constexpr int N64 = HW / 64, R64 = HW % 64;
#pragma unroll
    for (int i = 0; i < N64; ++i) {
        uint32_t v0[32], v1[32];
        tmem_ld32_nowait(taddr + 64u * i, v0);
        tmem_ld32_nowait(taddr + 64u * i + 32u, v1);
        tmem_wait_ld();
        epi_mid_store<32, EB, REMOTE>(v0, dst + (size_t)(64 * i / EPC) * PL, rdst + (uint32_t)(64 * i / EPC) * PL);
        epi_mid_store<32, EB, REMOTE>(v1, dst + (size_t)((64 * i + 32) / EPC) * PL, rdst + (uint32_t)((64 * i + 32) / EPC) * PL);
    }
    constexpr int c1 = N64 * 64;
    if constexpr (R64 >= 32) {
        uint32_t v0[32];
        tmem_ld32_nowait(taddr + c1, v0);
        tmem_wait_ld();
        epi_mid_store<32, EB, REMOTE>(v0, dst + (size_t)(c1 / EPC) * PL, rdst + (uint32_t)(c1 / EPC) * PL);
    }
    constexpr int c2 = c1 + (R64 >= 32 ? 32 : 0);
    if constexpr ((R64 % 32) >= 16) {
        uint32_t v0[16];
        tmem_ld16_nowait(taddr + c2, v0);
        tmem_wait_ld();
        epi_mid_store<16, EB, REMOTE>(v0, dst + (size_t)(c2 / EPC) * PL, rdst + (uint32_t)(c2 / EPC) * PL);
    }
    constexpr int c3 = c2 + ((R64 % 32) >= 16 ? 16 : 0);
    if constexpr ((R64 % 16) >= 8) {
        uint32_t v0[8];
        tmem_ld8_nowait(taddr + c3, v0);
        tmem_wait_ld();
        epi_mid_store<8, EB, REMOTE>(v0, dst + (size_t)(c3 / EPC) * PL, rdst + (uint32_t)(c3 / EPC) * PL);
    }
}

// any width that is a multiple of 8 (unusual channel counts)
template <int EB, bool REMOTE>
__device__ __forceinline__ void epi_mid_rt(int hw, uint32_t taddr, unsigned char* dst, uint32_t rdst) {
    constexpr int EPC = 16 / EB;
    constexpr uint32_t PL = T2_ROWS * 16;
    int c = 0;
    for (; c + 32 <= hw; c += 32)
        epi_mid<32, false, EB, REMOTE>(taddr + (uint32_t)c, dst + (size_t)(c / EPC) * PL, rdst + (uint32_t)(c / EPC) * PL);
    if (c + 16 <= hw) {
        epi_mid<16, false, EB, REMOTE>(taddr + (uint32_t)c, dst + (size_t)(c / EPC) * PL, rdst + (uint32_t)(c / EPC) * PL);
        c += 16;
    }
    if (c + 8 <= hw) epi_mid<8, false, EB, REMOTE>(taddr + (uint32_t)c, dst + (size_t)(c / EPC) * PL, rdst + (uint32_t)(c / EPC) * PL);
}

// max over W consecutive registers starting at v[O] (W = 8, 16 or 32), FMNMX3 tree
template <int O, int W>
__device__ __forceinline__ float max_run(const uint32_t (&v)[32]) {
    if constexpr (W == 1) {
        return __uint_as_float(v[O]);
    } else if constexpr (W == 2) {
        return fmaxf(__uint_as_float(v[O]), __uint_as_float(v[O + 1]));
    } else {
        float m = max3(__uint_as_float(v[O]), __uint_as_float(v[O + 1]), __uint_as_float(v[O + 2]));
#pragma unroll
        for (int j = 3; j + 1 < W; j += 2) m = max3(m, __uint_as_float(v[O + j]), __uint_as_float(v[O + j + 1]));
        if ((W & 1) == 0) m = fmaxf(m, __uint_as_float(v[O + W - 1]));
        return m;
    }
}

// emit(column of the centre's first row, its max) for every W-column centre of 32 loaded columns starting at c0
template <int W, int J = 0, class F>
__device__ __forceinline__ void emit_runs(const uint32_t (&v)[32], int c0, F&& emit) {
    if constexpr (J < 32 / W) {
        emit(c0 + J * W, max_run<J * W, W>(v));
        emit_runs<W, J + 1>(v, c0, emit);
    }
}

// GROUPS: tile pipelines per CTA; a pipeline is 128 * NH threads = NH (1 or 2) per tile row: thread (row, h) drains
// column part h of the row's TMEM lane in the mid-layer epilogues, gathers the 16-byte chunks kc = h (mod NH) of the
// row, and in the transposed last layer owns output channel `row` for 128 / NH of the tile's rows.  NH = 2 halves
// every warp's dependent chain per tile and doubles the warps, but duplicates the per-row bookkeeping (index load,
// frame arithmetic) -- it pays where a row is wide (chosen per shape in the launcher, TSMDET_MLP_NH overrides).
// SC = min(nsample, 32) in SA mode (8, 16 or 32).  DENSE: point-wise MLP over (B,C,n) inputs (features = source 0,
// src1 = source 1, concatenated along channels), no pooling.
// PF (SA mode): 16-byte feature chunks of a ROW that are prefetched INTO REGISTERS a whole tile ahead (4: <= 32
// channels, 16: <= 128 channels; half of them per thread); 0: rows of <= 4 channels read from the fp32 planes (a handful
// of registers, same one-tile-ahead schedule), or -- wider than 128 channels -- cp.async into the operand buffer behind
// the last MMA.  MINB: CTAs per SM the register allocation must allow.
// EB: bytes per operand element -- 2: bf16 operands (kind::f16), 4: tf32 operands (kind::tf32, fp32 bit patterns rounded
// to 10 mantissa bits; twice the shared memory and half the tensor rate, ~8x tighter than bf16).
// CL = 2: a tile is computed by a CLUSTER PAIR.  Each CTA holds half of every layer's output channels (half of the
// weights: a [131,128,128,256] MLP in tf32 is 278 KB of operands), both gather the tile's rows, each computes its half of a
// mid layer's activations and stores them into BOTH operand buffers (st.shared::cluster), and the transposed last layer
// splits by output-channel block.  Two cluster barriers per mid layer: "both MMAs have read the buffers" before the
// epilogues overwrite them, "both halves are written" before the next MMA.
template <int GROUPS, int SC, bool DENSE, int PF, int NH, int MINB, int EB, int CL = 1>
__global__ void __launch_bounds__(128 * NH * GROUPS, MINB)
    mlp_tc2_kernel(const __grid_constant__ SaMlpArgs a, const __grid_constant__ Tc2Plan pl,
                   const unsigned char* __restrict__ featT, const unsigned char* __restrict__ packed, const int fixed_tiles,
                   const int* __restrict__ cls) {
    constexpr int EPC = 16 / EB;  // operand elements per 16-byte chunk
    static_assert(CL == 1 || (GROUPS == 1 && NH == 1 && !DENSE), "cluster pairs: one tile pipeline of 128 threads per CTA");
    const uint32_t crank = CL == 2 ? cluster_ctarank() : 0u;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ __align__(8) uint64_t mma_bars[GROUPS];
    __shared__ __align__(8) uint64_t w_bar;
    __shared__ uint32_t tmem_base_s;

    constexpr int GT = 128 * NH;  // threads per tile group
    constexpr bool LEAN = GT * GROUPS * MINB >= 512;  // <= 128 registers per thread: fewer TMEM loads in flight
    constexpr int PFH = PF / NH;  // prefetch slots per thread
    const int grp = GROUPS == 1 ? 0 : (int)(threadIdx.x / GT);
    const int gt = threadIdx.x & (GT - 1);
    const int row = gt & 127;            // tile row (gather, mid-layer epilogues) / channel within a 128-block (last layer)
    const int h = NH == 1 ? 0 : gt >> 7;  // column part / chunk residue; warps 4h..4h+3 of the group, TMEM lane quadrant = warp & 3
    uint64_t& mma_bar = mma_bars[grp];
    auto group_sync = [&]() {
        if (GROUPS == 1) __syncthreads();
        else asm volatile("bar.sync %0, %1;" ::"r"(grp + 1), "n"(GT) : "memory");
    };
    const int S = a.s, M = a.m;
    const int M_tot = (int)(a.total_rows >> (31 - __clz(S)));  // centres B*M: the stride of the class lists
    const int log2s = 31 - __clz(S);
    const int nl = pl.nl;

    // width-class tiles: tt[k] = end of class k's tile range, tt[T2_MAX_CLS + k] = its number of centres
    const bool classed = !DENSE && pl.cls_off >= 0;
    int* const tt = reinterpret_cast<int*>(smem + (classed ? pl.cls_off : 0));
    if (classed) {
        if (threadIdx.x == 0) {
            int end = 0;
            for (int k = 0; k < pl.ncls; ++k) {
                const int n = cls[k];
                end += (n + (T2_ROWS >> k) - 1) >> (7 - k);
                tt[k] = end;
                tt[T2_MAX_CLS + k] = n;
            }
        }
        __syncthreads();
    }
    const int num_tiles = classed ? tt[pl.ncls - 1] : fixed_tiles;
    // A CTA whose tile groups all start past the last tile (width classes: the grid is sized for fixed-width tiles)
    // neither copies the weights nor allocates TMEM.  (Tile t runs on CTA t % G, see tile0 below.)
    const bool busy = (int)(blockIdx.x / CL) < num_tiles;

    // ---- one-time setup: weights + bias rows + ones operand arrive with ONE bulk copy (TMA engine); barriers; TMEM
    if (threadIdx.x == 0) {
        for (int g = 0; g < GROUPS; ++g) mbar_init(smem_u32(&mma_bars[g]), 1);
        mbar_init(smem_u32(&w_bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        if (busy) {
            mbar_arrive_expect_tx(smem_u32(&w_bar), (uint32_t)pl.packed_bytes);
            bulk_g2s(smem_u32(smem), packed + (size_t)crank * pl.packed_bytes, (uint32_t)pl.packed_bytes, smem_u32(&w_bar));
        }
    }
    if (busy && threadIdx.x < 32) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_s)),
                     "r"((uint32_t)pl.tmem_cols)
                     : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    if constexpr (CL == 2) cluster_sync_all();  // the peer CTA is resident before anything is stored into it
    // classed: tile -> its class k and the list position of its first centre
    auto tile_class = [&](int tile, int& first) {
        int k = 0;
        while (k + 1 < pl.ncls && tile >= tt[k]) ++k;
        first = (tile - (k > 0 ? tt[k - 1] : 0)) << (7 - k);
        return k;
    };
    bool weights_in = false;  // the weight image is awaited right before the first MMA: the first gather overlaps its copy
    auto wait_weights = [&]() {
        if (!weights_in) {
            const uint32_t bar = smem_u32(&w_bar);
            const long long t0 = clock64();
            unsigned spins = 0;
            while (!mbar_try_wait_cta(bar, 0))
                if ((++spins & 1023u) == 0 && clock64() - t0 > 4000000000LL) watchdog_trip(a.status, TSM_ERR_WATCHDOG);
            weights_in = true;
        }
    };
    const uint32_t d_tmem = tmem_base_s + (uint32_t)(grp * pl.grp_cols);
    // The MMAs are issued by one elected lane of the group's warp 0, from a warp-uniform branch with operands the
    // compiler knows to be uniform: issued from a divergent `if (thread == 0)`, every tcgen05.mma was wrapped in an
    // ELECT / 7 x R2UR waterfall loop (~19 instructions per MMA in the issuing thread, SASS).  The descriptors are
    // assembled from the plan (constant bank) and the shared-memory base in the uniform datapath -- no shared-memory
    // tables, no per-layer broadcasts (the path from the group barrier to the first MMA was ~100 instructions).
    const bool mma_warp = __shfl_sync(FULL, gt >> 5, 0) == 0;
    const uint32_t grp_u = __shfl_sync(FULL, (uint32_t)grp, 0);
    const uint32_t d_tmem_u = __shfl_sync(FULL, d_tmem, 0);
    constexpr uint32_t DESC_HI = (128u >> 4) | (1u << 14);  // SBO = 128 B, descriptor version 1 (bit 46)
    auto desc_lo = [](uint32_t addr, uint32_t lbo) { return ((addr >> 4) & 0x3fffu) | (((lbo >> 4) & 0x3fffu) << 16); };
    auto umma = [](uint32_t d, uint64_t ad, uint64_t bd, uint32_t idesc, uint32_t acc) {
        if constexpr (EB == 2) umma_bf16(d, ad, bd, idesc, acc);
        else umma_tf32(d, ad, bd, idesc, acc);
    };
    const uint32_t t_lane = d_tmem + ((uint32_t)(row & ~31) << 16);  // this warp's 32 TMEM lanes
    const uint32_t a_smem = smem_u32(smem + pl.a_off + grp * pl.a_bytes);
    unsigned char* const a_ptr = smem + pl.a_off + grp * pl.a_bytes;
    unsigned char* const a_row = a_ptr + row * 16;  // this thread's row inside every 16-byte chunk plane
    uint32_t phase = 0;
    const int cout_last = a.ch[nl];
    const int nchunk0 = pl.K[0] / EPC;
    // tile t -> CTA t % G, group (t / G) % GROUPS (G = CTAs, or pairs): fewer tiles than groups (width classes) still
    // land on as many SMs as there are tiles; both CTAs of a pair walk the same tiles
    const int tile0 = grp * (int)(gridDim.x / CL) + (int)(blockIdx.x / CL), tile_step = (gridDim.x / CL) * GROUPS;

    // SA mode: the neighbour index and the hit count of this thread's row are LOADED one tile ahead and only looked at
    // when the next gather is issued; the coordinates are loaded when the gather is issued and only looked at when it
    // is finished -- no load is consumed where it is issued.
    // Classed tiles: row r of a class-k tile is slot r % 2^k of centre list[first + r / 2^k] (cg_raw, -1 past the
    // class's end); its neighbour index is loaded behind the list entry in the same prefetch.
    int id_raw = 0, cnt_raw = 1, cg_raw = -1;
    auto prefetch_row = [&](int tile) {
        if constexpr (!DENSE) {
            id_raw = 0;
            cnt_raw = 0;  // rows past the end are masked
            cg_raw = -1;
            if (classed) {
                if (tile < num_tiles) {
                    int first;
                    const int k = tile_class(tile, first);
                    const int pos = first + (row >> k);
                    if (pos < tt[T2_MAX_CLS + k]) {
                        const int v = __ldg(cls + T2_CLS_LIST + (size_t)k * M_tot + pos);
                        cg_raw = v >= 0 ? v : ~v;
                        cnt_raw = v >= 0 ? 1 : 0;
                        id_raw = __ldg(a.idx + (size_t)cg_raw * S + (row & ((1 << k) - 1)));
                    }
                }
            } else if (tile < num_tiles) {
                const long long g = (long long)tile * T2_ROWS + row;
                if (g < a.total_rows) {
                    id_raw = __ldg(a.idx + g);
                    cnt_raw = a.idx_cnt ? __ldg(a.idx_cnt + (g >> log2s)) : 1;  // <= 0: empty ball -> zero input row
                }
            }
        }
    };
    // load_row(tile): every load of this thread's chunks of the row (parity h) -- coordinates, and the features as PFH
    // register chunks / fp32 planes / cp.async -- is ISSUED; store_row(): what arrived in registers goes to the operand
    // buffer.  With PF > 0 or planar rows, load_row(i+1) is issued right after store_row(i), so the loads have a whole
    // tile of compute to land; the cp.async form needs the buffer itself and is issued behind tile i's last MMA.
    float pend_p[3] = {0.f, 0.f, 0.f}, pend_q[3] = {0.f, 0.f, 0.f}, pend_f[4] = {0.f, 0.f, 0.f, 0.f};
    uint4 pf_row[PFH > 0 ? PFH : 1];
    bool pend_live = false;
    const uint32_t a_row_s = a_smem + (uint32_t)row * 16u;
    const bool planar = PF == 0 && featT == nullptr && a.c_feat > 0;  // <= 4 feature channels: read straight from (B,C,N) fp32
    const bool own_xyz = pl.xyz_chunk >= 0 && (NH == 1 || (pl.xyz_chunk & 1) == h);
    // Register-prefetched feature chunks are split between the two threads of a row (NH == 2) or the two CTAs of a pair
    // (CL == 2: each gathers every other chunk and stores it into BOTH operand buffers -- half the gather traffic, and
    // the one-tile-ahead register path instead of cp.async for rows of up to 32 chunks)
    constexpr int CST = NH * CL;                    // chunk stride of this thread's slots
    const int coff = CL == 2 ? (int)crank : h;      // its first chunk
    const uint32_t a_row_peer = CL == 2 ? mapa_u32(a_row_s, crank ^ 1u) : 0u;
    constexpr bool kEarly = PF > 0;  // (planar rows are early too: decided at run time)
    auto load_row = [&](int tile) {
        if constexpr (!DENSE) {
            const long long g = (long long)tile * T2_ROWS + row;
            const int id = id_raw;
            const bool live = cnt_raw > 0;
            pend_live = live;
            const long long cpi = classed ? (cg_raw >= 0 ? cg_raw : 0) : (g < a.total_rows ? (g >> log2s) : 0);  // S is a power of two; B*M < 2^31 (launcher)
            const int b = (int)((unsigned)cpi / (unsigned)M);
            const size_t prow = (size_t)b * a.n + id;
            if (own_xyz && live) {
                const float* p = a.xyz + prow * 3;
                const float* q = a.new_xyz + (size_t)cpi * 3;
#pragma unroll
                for (int k = 0; k < 3; ++k) {
                    pend_p[k] = __ldg(p + k);
                    pend_q[k] = __ldg(q + k);
                }
            }
            if (planar) {
                if (live && h == 0) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
                        if (k < a.c_feat) pend_f[k] = __ldg(a.features + ((size_t)b * a.c_feat + k) * a.n + id);
                }
            } else if constexpr (PF > 0) {
                const int fchunks = pl.cp / EPC;
                const uint4* frow = reinterpret_cast<const uint4*>(featT + prow * pl.cp * EB);
#pragma unroll
                for (int j = 0; j < PFH; ++j) {
                    pf_row[j] = make_uint4(0u, 0u, 0u, 0u);
                    if (live && CST * j + coff < fchunks) pf_row[j] = __ldg(frow + CST * j + coff);
                }
            } else if (featT != nullptr) {
                const int fchunks = pl.cp / EPC;
                const uint4* frow = reinterpret_cast<const uint4*>(featT + prow * pl.cp * EB);
                const int nbytes = live ? 16 : 0;  // src-size 0: the 16 destination bytes are zero-filled, nothing is read
                for (int kc = h; kc < fchunks; kc += NH)
                    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(a_row_s + (uint32_t)kc * (T2_ROWS * 16)),
                                 "l"(frow + kc), "r"(nbytes)
                                 : "memory");
                asm volatile("cp.async.commit_group;" ::: "memory");
            }
        }
    };
    auto store_row = [&]() {
        if constexpr (!DENSE) {
            const int fchunks = (planar || featT == nullptr) ? 0 : (pl.cp / EPC);
            if constexpr (PF > 0) {
#pragma unroll
                for (int j = 0; j < PFH; ++j) {
                    if (CST * j + coff < fchunks) {
                        *reinterpret_cast<uint4*>(a_row + (size_t)(CST * j + coff) * (T2_ROWS * 16)) = pf_row[j];
                        if constexpr (CL == 2) st_cluster_v4(a_row_peer + (uint32_t)(CST * j + coff) * (T2_ROWS * 16), pf_row[j]);
                    }
                }
            }
            // this thread's chunks behind the features: coordinates, planar features, zero padding
            for (int kc = fchunks + (NH == 2 ? ((fchunks ^ h) & 1) : 0); kc < nchunk0; kc += NH) {
                uint4 v = make_uint4(0u, 0u, 0u, 0u);
                if (pend_live) {
                    if (kc == pl.xyz_chunk) {
                        const float dx = __fsub_rn(pend_p[0], pend_q[0]), dy = __fsub_rn(pend_p[1], pend_q[1]), dz = __fsub_rn(pend_p[2], pend_q[2]);
                        if constexpr (EB == 2) {
                            v.x = pack_bf16(dx, dy);
                            v.y = pack_bf16(dz, 0.f);
                        } else {
                            v = make_uint4(to_tf32(dx), to_tf32(dy), to_tf32(dz), 0u);
                        }
                    } else if (planar && kc == 0) {
                        const float f1 = a.c_feat > 1 ? pend_f[1] : 0.f, f2 = a.c_feat > 2 ? pend_f[2] : 0.f, f3 = a.c_feat > 3 ? pend_f[3] : 0.f;
                        if constexpr (EB == 2) {
                            v.x = pack_bf16(pend_f[0], f1);
                            v.y = pack_bf16(f2, f3);
                        } else {
                            v = make_uint4(to_tf32(pend_f[0]), to_tf32(f1), to_tf32(f2), to_tf32(f3));
                        }
                    }
                }
                *reinterpret_cast<uint4*>(a_row + (size_t)kc * (T2_ROWS * 16)) = v;
            }
            if (PF == 0 && !planar) asm volatile("cp.async.wait_all;" ::: "memory");
        }
    };
    auto wait_mma = [&]() {
        const uint32_t bar = smem_u32(&mma_bar);
        if (!mbar_try_wait_cta(bar, phase)) {  // try_wait suspends the thread for a hardware time slice per call
            const long long t0 = clock64();
            unsigned spins = 0;
            while (!mbar_try_wait_cta(bar, phase))
                if ((++spins & 1023u) == 0 && clock64() - t0 > 4000000000LL) watchdog_trip(a.status, TSM_ERR_WATCHDOG);
        }
        phase ^= 1u;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };

#ifdef MLP_PROF
    const bool prof_on = blockIdx.x == 0 && grp == 0 && gt == 32;
    long long prof_acc[8] = {0, 0, 0, 0, 0, 0, 0, 0}, prof_t = clock64(), prof_tiles = 0, prof_issue = 0;
    const long long prof_t0 = prof_t;
#endif
    const bool early = kEarly || planar;
    prefetch_row(tile0);
    if (tile0 < num_tiles) load_row(tile0);
    prefetch_row(tile0 + tile_step);

    for (int tile = tile0; tile < num_tiles; tile += tile_step) {
        // ------------------------------------------------------------------ layer-0 operand
        if constexpr (!DENSE) {
            store_row();
        } else {
            // dense: channel c of row g = src0[b, c, i] (c < c_feat) | src1[b, c - c_feat, i]; coalesced over threads;
            // thread (row, h) builds the 32-channel blocks h (mod NH)
            const long long g = (long long)tile * T2_ROWS + row;  // this thread's global row
            const bool rv = g < a.total_rows;
            const int b = rv ? (int)(g / a.n) : 0;
            const int i = rv ? (int)(g - (long long)b * a.n) : 0;
            const float* s0 = a.features + (size_t)b * a.c_feat * a.n + i;
            const float* s1 = a.src1 ? a.src1 + (size_t)b * a.c1 * a.n + i : nullptr;
            const int ctot = a.c_feat + a.c1;
            constexpr int CPI = 32 / EPC;  // chunks per 32-channel block
            for (int kc0 = CPI * h; kc0 < nchunk0; kc0 += CPI * NH) {
                float x[32];
#pragma unroll
                for (int u = 0; u < 32; ++u) {
                    const int c = kc0 * EPC + u;
                    x[u] = 0.f;
                    if (rv && c < ctot) x[u] = c < a.c_feat ? __ldg(s0 + (size_t)c * a.n) : __ldg(s1 + (size_t)(c - a.c_feat) * a.n);
                }
#pragma unroll
                for (int u = 0; u < CPI; ++u) {
                    if (kc0 + u < nchunk0) {
                        uint4 v;
                        if constexpr (EB == 2)
                            v = make_uint4(pack_bf16(x[8 * u], x[8 * u + 1]), pack_bf16(x[8 * u + 2], x[8 * u + 3]),
                                           pack_bf16(x[8 * u + 4], x[8 * u + 5]), pack_bf16(x[8 * u + 6], x[8 * u + 7]));
                        else
                            v = make_uint4(to_tf32(x[4 * u]), to_tf32(x[4 * u + 1]), to_tf32(x[4 * u + 2]), to_tf32(x[4 * u + 3]));
                        *reinterpret_cast<uint4*>(a_row + (size_t)(kc0 + u) * (T2_ROWS * 16)) = v;
                    }
                }
            }
        }
        MPROF(0);  // operand build
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        wait_weights();
        if constexpr (CL == 2) {
            asm volatile("fence.proxy.async;" ::: "memory");  // local and remote stores of the operand
            cluster_sync_all();                                // both CTAs' halves of the gathered rows are in both buffers
        } else {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            group_sync();
        }
        MPROF(1);  // fence + barrier

        // ------------------------------------------------------------------ layers 0 .. nl-2: D[row, cout] in TMEM
        for (int l = 0; l + 1 < nl; ++l) {
            const int Np = pl.Npad[l];
            if (mma_warp) {  // warp-uniform branch, uniform operands: the descriptors live in uniform registers
#ifdef MLP_PROF
                const long long ti0 = clock64();
#endif
                if constexpr (CL == 2) asm volatile("fence.proxy.async;" ::: "memory");  // the peer's stores -> async proxy
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                // act (A, M = 128 rows) x W_l (B, N = Np); per K step of 16 only the start-address fields advance;
                // last step: ones (A) x [bias_hi, bias_lo] rows -- the bias lands in the accumulator
                const uint32_t sbase = smem_u32(smem);
                const uint32_t a_lo = desc_lo(sbase + (uint32_t)pl.a_off + grp_u * (uint32_t)pl.a_bytes, T2_ROWS * 16);  // LBO = 128 rows x 16 B
                const uint32_t o_lo = desc_lo(sbase + (uint32_t)pl.ones_off, T2_ROWS * 16);
                const uint32_t w_lo = desc_lo(sbase + (uint32_t)pl.w_off[l], (uint32_t)Np * 16);  // LBO = Npad rows x 16 B
                const uint32_t idesc = EB == 2 ? instr_desc_bf16_m128(Np) : instr_desc_tf32_m128(Np), wstep = (2u * (uint32_t)Np * 16u) >> 4;
                constexpr uint32_t a_hi = DESC_HI, o_hi = DESC_HI, w_hi = DESC_HI;
                const int nk = pl.K[l] / (2 * EPC);
                if (elect_one()) {
                    uint32_t ad = a_lo, wd = w_lo;
                    for (int kk = 0; kk < nk; ++kk) {
                        umma(d_tmem_u, desc64(ad, a_hi), desc64(wd, w_hi), idesc, kk > 0 ? 1u : 0u);
                        ad += (2u * T2_ROWS * 16u) >> 4;
                        wd += wstep;
                    }
                    umma(d_tmem_u, desc64(o_lo, o_hi), desc64(wd, w_hi), idesc, 1u);
                    umma_commit(smem_u32(&mma_bar));
                }
                __syncwarp();
#ifdef MLP_PROF
                prof_issue += clock64() - ti0;
#endif
            }
            wait_mma();
            MPROF(2);  // mid-layer MMA issue + wait
            if constexpr (CL == 2) cluster_sync_all();  // both CTAs' MMAs have read their operand buffers
            // ReLU -> bf16 / tf32 -> next layer's A operand (written over the consumed one); thread = (row, column part h);
            // in a pair this CTA's columns are activation channels [crank * Np, (crank + 1) * Np)
            const int hw = Np / NH;
            const uint32_t ta = t_lane + (uint32_t)(h * hw);
            const uint32_t poff = (uint32_t)(((int)crank * Np + h * hw) / EPC) * (T2_ROWS * 16);
            unsigned char* const dst = a_row + poff;
            const uint32_t rdst = CL == 2 ? mapa_u32(a_row_s + poff, crank ^ 1u) : 0u;
            constexpr bool RM = CL == 2;
            switch (hw) {
                case 8: epi_mid<8, false, EB, RM>(ta, dst, rdst); break;
                case 16: epi_mid<16, false, EB, RM>(ta, dst, rdst); break;
                case 32: epi_mid<32, false, EB, RM>(ta, dst, rdst); break;
                case 64: epi_mid<64, LEAN, EB, RM>(ta, dst, rdst); break;
                case 128: epi_mid<128, LEAN, EB, RM>(ta, dst, rdst); break;
                case 256: epi_mid<256, LEAN, EB, RM>(ta, dst, rdst); break;
                default: epi_mid_rt<EB, RM>(hw, ta, dst, rdst); break;
            }
            MPROF(3);  // mid-layer epilogue
            asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
            if constexpr (CL == 2) {
                asm volatile("fence.proxy.async;" ::: "memory");  // local and remote stores
                cluster_sync_all();                                // both halves of the activations are in both buffers
            } else {
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                group_sync();
            }
            MPROF(1);
        }

        // ------------------------------------------------------------------ last layer, transposed: D^T[cout, row]
        {
            const int l = nl - 1;
            if (mma_warp) {
                if constexpr (CL == 2) asm volatile("fence.proxy.async;" ::: "memory");
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                // W_last block mb (A, M = 128 channels) x act (B, N = 128 rows)
                const uint32_t sbase = smem_u32(smem);
                const uint32_t a_lo = desc_lo(sbase + (uint32_t)pl.a_off + grp_u * (uint32_t)pl.a_bytes, T2_ROWS * 16);
                const uint32_t w_lo = desc_lo(sbase + (uint32_t)pl.w_off[l], (uint32_t)pl.Npad[l] * 16);
                const uint32_t idesc = EB == 2 ? instr_desc_bf16_m128(T2_ROWS) : instr_desc_tf32_m128(T2_ROWS), wstep = (2u * (uint32_t)pl.Npad[l] * 16u) >> 4;
                constexpr uint32_t a_hi = DESC_HI, w_hi = DESC_HI;
                const int nk = pl.K[l] / (2 * EPC);
                if (elect_one()) {
                    for (int mb = 0; mb < pl.mb; ++mb) {
                        uint32_t ad = a_lo, wd = w_lo + (uint32_t)((mb * T2_ROWS * 16) >> 4);
                        for (int kk = 0; kk < nk; ++kk) {
                            umma(d_tmem_u + (uint32_t)(mb * T2_ROWS), desc64(wd, w_hi), desc64(ad, a_hi), idesc, kk > 0 ? 1u : 0u);
                            ad += (2u * T2_ROWS * 16u) >> 4;
                            wd += wstep;
                        }
                    }
                    umma_commit(smem_u32(&mma_bar));
                }
                __syncwarp();
            }
            // The next tile's row loads are issued here: they fly during the last MMA and the pooling epilogue and are
            // consumed by the next store_row().  (Issued at the top of the tile, the prefetched registers were live across
            // the mid-layer epilogues and ptxas spilled them right behind the loads -- STL stalls on the load, ncu.)
            if (early) {
                if (tile + tile_step < num_tiles) load_row(tile + tile_step);
                prefetch_row(tile + 2 * tile_step);
            }
            MPROF(4);  // next tile's loads issued
            wait_mma();
            if constexpr (CL == 2) cluster_sync_all();  // both CTAs' last MMAs have read the buffers the next gather overwrites
            MPROF(5);  // last MMA wait
            if (!early) {  // cp.async rows: the operand buffer is free again, the copies land during the epilogue below
                if (tile + tile_step < num_tiles) load_row(tile + tile_step);
                prefetch_row(tile + 2 * tile_step);
            }
            const float* bs = reinterpret_cast<const float*>(smem + pl.b_off);
            constexpr int PW = T2_ROWS / NH;                      // tile rows (TMEM columns) per thread
            const uint32_t t_part = t_lane + (uint32_t)(PW * h);  // this thread's columns of every channel block

            if constexpr (!DENSE) {
                // thread = (output channel, half of the tile's rows): max over the S columns of a centre in registers,
                // then bias + ReLU once per centre (both monotone: max(relu(x+b)) == relu(max(x)+b) bit for bit)
                const int cpt = T2_ROWS >> log2s;  // centres per tile
                const unsigned cbase = (unsigned)tile * (unsigned)cpt;
                const unsigned ctot = (unsigned)(a.total_rows >> log2s);
                const unsigned b0 = cbase / (unsigned)M, p0 = cbase - b0 * (unsigned)M;
                const int cpo = (cout_last + EPC - 1) / EPC * EPC;  // width of the operand-type row copy (zero padded)
                using RowT = std::conditional_t<EB == 2, __nv_bfloat16, float>;
                auto to_row = [](float y) -> RowT {
                    if constexpr (EB == 2) return __float2bfloat16_rn(y);
                    else return __uint_as_float(to_tf32(y));
                };
                const bool full = pl.whole_tiles && cbase + (unsigned)cpt <= ctot;  // every centre valid, one frame
                float part0 = 0.f, part1 = 0.f;  // NH == 2, S == 128: this half's maximum per channel block
                auto pool = [&](auto full_tag) {
                    constexpr bool FULL = decltype(full_tag)::value;
                    for (int mb = 0; mb < pl.mb; ++mb) {
                        const int ch = (mb + (int)crank) * T2_ROWS + row;  // (a pair: CTA `crank` owns channel block `crank`)
                        const float bias = bs[mb * T2_ROWS + row];
                        const bool ch_ok = ch < cout_last;
                        float* const obase = a.out + ((size_t)b0 * a.out_ctot + a.out_c0 + (ch_ok ? ch : 0)) * M + p0;
                        RowT* const tbase = reinterpret_cast<RowT*>(a.out_t) + (size_t)cbase * cpo + ch;
                        const bool o_ok = a.out != nullptr && ch_ok;
                        const bool t_ok = a.out_t != nullptr && ch < cpo;
                        auto emit = [&](int ci, float m) {
                            const float y = ch_ok ? fmaxf(__fadd_rn(m, bias), 0.f) : 0.f;
                            if constexpr (FULL) {
                                if (o_ok) obase[ci] = y;
                                // (B,M,cpo) bf16 rows for the next layer's gather: a warp writes 32 consecutive channels
                                if (t_ok) tbase[(size_t)ci * cpo] = to_row(y);
                            } else {
                                const unsigned cg = cbase + (unsigned)ci;
                                if (cg < ctot) {
                                    if (o_ok) {  // a tile may straddle two frames
                                        const unsigned b2 = cg / (unsigned)M, p2 = cg - b2 * (unsigned)M;
                                        a.out[((size_t)b2 * a.out_ctot + a.out_c0 + ch) * M + p2] = y;
                                    }
                                    if (t_ok) tbase[(size_t)ci * cpo] = to_row(y);
                                }
                            }
                        };
                        if ((mb + (int)crank) * T2_ROWS + (row & ~31) >= (cpo > cout_last ? cpo : cout_last)) continue;  // warp-uniform: padding channels
                        float run = 0.f;
#pragma unroll 1
                        for (int cb = 0; cb < PW; cb += 64) {
                            const int c0 = PW * h + cb;  // first tile row of this batch
                            uint32_t v0[32], v1[32];
                            tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb), v0);
                            if constexpr (LEAN && SC < 32) {  // half the registers: the first 32 columns are emitted before the second load
                                tmem_wait_ld();
                                if constexpr (SC == 16) {
                                    emit((c0 >> 4) + 0, max_run<0, 16>(v0));
                                    emit((c0 >> 4) + 1, max_run<16, 16>(v0));
                                } else {
                                    emit((c0 >> 3) + 0, max_run<0, 8>(v0));
                                    emit((c0 >> 3) + 1, max_run<8, 8>(v0));
                                    emit((c0 >> 3) + 2, max_run<16, 8>(v0));
                                    emit((c0 >> 3) + 3, max_run<24, 8>(v0));
                                }
                                tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb + 32), v0);
                                tmem_wait_ld();
                                if constexpr (SC == 16) {
                                    emit((c0 >> 4) + 2, max_run<0, 16>(v0));
                                    emit((c0 >> 4) + 3, max_run<16, 16>(v0));
                                } else {
                                    emit((c0 >> 3) + 4, max_run<0, 8>(v0));
                                    emit((c0 >> 3) + 5, max_run<8, 8>(v0));
                                    emit((c0 >> 3) + 6, max_run<16, 8>(v0));
                                    emit((c0 >> 3) + 7, max_run<24, 8>(v0));
                                }
                                continue;
                            }
                            float m0 = 0.f, m1 = 0.f;
                            if constexpr (LEAN && SC == 32) {  // one load in flight, the same registers twice
                                tmem_wait_ld();
                                m0 = max_run<0, 32>(v0);
                                tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb + 32), v0);
                                tmem_wait_ld();
                                m1 = max_run<0, 32>(v0);
                            } else {
                                tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb + 32), v1);
                                tmem_wait_ld();
                                if constexpr (SC == 32) {
                                    m0 = max_run<0, 32>(v0);
                                    m1 = max_run<0, 32>(v1);
                                }
                            }
                            if constexpr (SC == 32) {
                                // S = 32, 64 or 128: a 32-column chunk lies inside one centre
                                if (S == 32) {
                                    emit(c0 >> 5, m0);
                                    emit((c0 >> 5) + 1, m1);
                                } else if (S == 64) {
                                    emit(c0 >> 6, fmaxf(m0, m1));
                                } else if (NH == 1) {  // S == 128, one thread per channel
                                    run = cb == 0 ? fmaxf(m0, m1) : max3(run, m0, m1);
                                    if (cb == 64) emit(0, run);
                                } else {  // S == 128: the two halves of a channel meet in shared memory (below)
                                    if (mb == 0) part0 = fmaxf(m0, m1);
                                    else part1 = fmaxf(m0, m1);
                                }
                            } else if constexpr (SC == 16) {
                                emit((c0 >> 4) + 0, max_run<0, 16>(v0));
                                emit((c0 >> 4) + 1, max_run<16, 16>(v0));
                                emit((c0 >> 4) + 2, max_run<0, 16>(v1));
                                emit((c0 >> 4) + 3, max_run<16, 16>(v1));
                            } else {  // SC == 8
                                emit((c0 >> 3) + 0, max_run<0, 8>(v0));
                                emit((c0 >> 3) + 1, max_run<8, 8>(v0));
                                emit((c0 >> 3) + 2, max_run<16, 8>(v0));
                                emit((c0 >> 3) + 3, max_run<24, 8>(v0));
                                emit((c0 >> 3) + 4, max_run<0, 8>(v1));
                                emit((c0 >> 3) + 5, max_run<8, 8>(v1));
                                emit((c0 >> 3) + 6, max_run<16, 8>(v1));
                                emit((c0 >> 3) + 7, max_run<24, 8>(v1));
                            }
                        }
                    }
                };
                int xk = log2s;  // log2 of this tile's rows per centre
                if (classed) {
                    // one 32-column load at a time; centre j of a class-k tile is list entry first + j, its rows are
                    // columns j << k ..
                    int first;
                    xk = tile_class(tile, first);
                    const int* const lst = cls + T2_CLS_LIST + (size_t)xk * M_tot + first;
                    const int nlst = tt[T2_MAX_CLS + xk] - first;
                    for (int mb = 0; mb < pl.mb; ++mb) {
                        const int ch = (mb + (int)crank) * T2_ROWS + row;
                        const float bias = bs[mb * T2_ROWS + row];
                        const bool ch_ok = ch < cout_last;
                        const bool o_ok = a.out != nullptr && ch_ok;
                        const bool t_ok = a.out_t != nullptr && ch < cpo;
                        auto emit = [&](int c, float m) {  // c: tile column of the centre's first row
                            if ((c >> xk) >= nlst) return;  // past the end of the class
                            const int v = __ldg(lst + (c >> xk));
                            const int cg = v >= 0 ? v : ~v;
                            const float y = ch_ok ? fmaxf(__fadd_rn(m, bias), 0.f) : 0.f;
                            if (o_ok) {
                                const unsigned b2 = (unsigned)cg / (unsigned)M, p2 = (unsigned)cg - b2 * (unsigned)M;
                                a.out[((size_t)b2 * a.out_ctot + a.out_c0 + ch) * M + p2] = y;
                            }
                            if (t_ok) reinterpret_cast<RowT*>(a.out_t)[(size_t)cg * cpo + ch] = to_row(y);
                        };
                        if ((mb + (int)crank) * T2_ROWS + (row & ~31) >= (cpo > cout_last ? cpo : cout_last)) continue;  // warp-uniform: padding channels
                        float run = 0.f;
#pragma unroll 1
                        for (int cb = 0; cb < PW; cb += 32) {
                            const int c0 = PW * h + cb;
                            uint32_t v[32];
                            tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb), v);
                            tmem_wait_ld();
                            switch (xk) {
                                case 0: emit_runs<1>(v, c0, emit); break;
                                case 1: emit_runs<2>(v, c0, emit); break;
                                case 2: emit_runs<4>(v, c0, emit); break;
                                case 3: emit_runs<8>(v, c0, emit); break;
                                case 4: emit_runs<16>(v, c0, emit); break;
                                default: {  // 32, 64 or 128 rows per centre: the 32 columns lie inside one centre
                                    const int w = 1 << xk;
                                    const float m = max_run<0, 32>(v);
                                    run = (cb == 0 || (c0 & (w - 1)) == 0) ? m : fmaxf(run, m);  // (a half: from its first column)
                                    if (((c0 + 32) & (w - 1)) == 0 && w <= PW) emit(c0 + 32 - w, run);
                                }
                            }
                        }
                        if (mb == 0) part0 = run;  // 128 rows per centre, NH == 2: this half's maximum (below)
                        else part1 = run;
                    }
                } else if (full) {
                    pool(std::true_type{});
                } else {
                    pool(std::false_type{});
                }
                if (NH == 2 && SC == 32 && xk == 7) {  // uniform; the next write of xbuf lies behind the next tile's barriers
                    float* const xbuf = reinterpret_cast<float*>(smem + pl.x_off) + grp * (2 * T2_ROWS);
                    if (h == 1) {
                        xbuf[row] = part0;
                        xbuf[T2_ROWS + row] = part1;
                    }
                    group_sync();
                    int cg = cbase < ctot ? (int)cbase : -1;  // one centre per tile
                    if (classed) {
                        int first;
                        tile_class(tile, first);
                        const int v = __ldg(cls + T2_CLS_LIST + (size_t)7 * M_tot + first);
                        cg = v >= 0 ? v : ~v;
                    }
                    if (h == 0 && cg >= 0) {
                        const unsigned b2 = (unsigned)cg / (unsigned)M, p2 = (unsigned)cg - b2 * (unsigned)M;
                        for (int mb = 0; mb < pl.mb; ++mb) {
                            const int ch = mb * T2_ROWS + row;  // (NH == 2 excludes cluster pairs)
                            const bool ch_ok = ch < cout_last;
                            const float m = fmaxf(mb == 0 ? part0 : part1, xbuf[mb * T2_ROWS + row]);
                            const float y = ch_ok ? fmaxf(__fadd_rn(m, bs[ch]), 0.f) : 0.f;
                            if (a.out != nullptr && ch_ok) a.out[((size_t)b2 * a.out_ctot + a.out_c0 + ch) * M + p2] = y;
                            if (a.out_t != nullptr && ch < cpo) reinterpret_cast<RowT*>(a.out_t)[(size_t)cg * cpo + ch] = to_row(y);
                        }
                    }
                }
                // no barrier here: the next tile's MMA is issued after the barrier that follows store_row()
            } else {
                // dense: thread = (output channel, half): 64 columns = 64 consecutive rows (points) of the tile
                const long long g0 = (long long)tile * T2_ROWS;
                const int b0 = (int)(g0 / a.n);
                const int i0 = (int)(g0 - (long long)b0 * a.n);
                const bool whole = (i0 + T2_ROWS <= a.n) && (g0 + T2_ROWS <= a.total_rows);  // one batch entry, full tile
                for (int mb = 0; mb < pl.mb; ++mb) {
                    const int ch = mb * T2_ROWS + row;
                    const float bias = bs[ch];
                    const bool ch_ok = ch < cout_last;
                    if (mb * T2_ROWS + (row & ~31) >= cout_last) continue;  // warp-uniform: padding channels
                    float* const orow = a.out + ((size_t)b0 * a.out_ctot + a.out_c0 + (ch_ok ? ch : 0)) * a.n + i0 + PW * h;
                    const bool vec = whole && ((reinterpret_cast<uintptr_t>(orow) & 15u) == 0);
#pragma unroll 1
                    for (int cb = 0; cb < PW; cb += 64) {
                        uint32_t v0[32], v1[32];
                        tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb), v0);
                        tmem_ld32_nowait(t_part + (uint32_t)(mb * T2_ROWS + cb + 32), v1);
                        tmem_wait_ld();
                        if (!ch_ok) continue;
                        if (vec) {
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                float4 o;
                                o.x = fmaxf(__uint_as_float(v0[4 * q + 0]) + bias, 0.f);
                                o.y = fmaxf(__uint_as_float(v0[4 * q + 1]) + bias, 0.f);
                                o.z = fmaxf(__uint_as_float(v0[4 * q + 2]) + bias, 0.f);
                                o.w = fmaxf(__uint_as_float(v0[4 * q + 3]) + bias, 0.f);
                                *reinterpret_cast<float4*>(orow + cb + 4 * q) = o;
                            }
#pragma unroll
                            for (int q = 0; q < 8; ++q) {
                                float4 o;
                                o.x = fmaxf(__uint_as_float(v1[4 * q + 0]) + bias, 0.f);
                                o.y = fmaxf(__uint_as_float(v1[4 * q + 1]) + bias, 0.f);
                                o.z = fmaxf(__uint_as_float(v1[4 * q + 2]) + bias, 0.f);
                                o.w = fmaxf(__uint_as_float(v1[4 * q + 3]) + bias, 0.f);
                                *reinterpret_cast<float4*>(orow + cb + 32 + 4 * q) = o;
                            }
                        } else {
#pragma unroll
                            for (int j = 0; j < 64; ++j) {
                                const long long g2 = g0 + PW * h + cb + j;
                                if (g2 < a.total_rows) {
                                    const int b2 = (int)(g2 / a.n);
                                    const int i2 = (int)(g2 - (long long)b2 * a.n);
                                    const float x = __uint_as_float(j < 32 ? v0[j & 31] : v1[j & 31]);
                                    a.out[((size_t)b2 * a.out_ctot + a.out_c0 + ch) * a.n + i2] = fmaxf(x + bias, 0.f);
                                }
                            }
                        }
                    }
                }
            }
        }
#ifdef MLP_PROF
        MPROF(6);  // pooling / output epilogue
        ++prof_tiles;
#endif
    }

#ifdef MLP_PROF
    if (blockIdx.x == 0 && grp == 0 && gt == 0 && tile0 < num_tiles)
        printf("   issuing warp: barrier exit -> commit issued, mid layers, cycles per tile: %lld\n",
               prof_issue / ((num_tiles - tile0 + tile_step - 1) / tile_step));
    if (prof_on && prof_tiles > 0)
        printf("mlp_tc2<G%d,SC%d,D%d,PF%d,NH%d> tiles/group %lld cycles/tile: total %lld | build %lld fence+bar %lld mid-mma-wait %lld mid-epi %lld "
               "issue-loads %lld last-mma-wait %lld pool %lld\n",
               GROUPS, SC, (int)DENSE, PF, NH, prof_tiles, (clock64() - prof_t0) / prof_tiles, prof_acc[0] / prof_tiles,
               prof_acc[1] / prof_tiles, prof_acc[2] / prof_tiles, prof_acc[3] / prof_tiles, prof_acc[4] / prof_tiles,
               prof_acc[5] / prof_tiles, prof_acc[6] / prof_tiles);
#endif
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if constexpr (CL == 2) cluster_sync_all();  // no CTA leaves while its peer may still store into it
    if (busy && threadIdx.x < 32) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base_s), "r"((uint32_t)pl.tmem_cols)
                     : "memory");
    }
}

}  // namespace tsm

static int round_up2(int v, int m) { return (v + m - 1) / m * m; }

// Shapes this kernel takes and the shared-memory / TMEM plan for them.  TSM_ERR_INVALID otherwise (the caller falls
// back to sa_mlp_tc.cu / the fp32 kernel).
static int tc2_plan_cl(const tsm::SaMlpArgs& a, long long centres, int dense, int eb, int cl, tsm::Tc2Plan* out, int* groups_out) {
    using namespace tsm;
    const int S = a.s;
    if (eb != 2 && eb != 4) return TSM_ERR_INVALID;
    if (cl != 1 && (cl != 2 || dense || S == T2_ROWS)) return TSM_ERR_INVALID;  // pairs: SA scales, 128 threads per CTA
    const int epc = 16 / eb, ks = 2 * epc;  // operand elements per 16-byte chunk / per K step
    if (a.num_layers < 1 || a.num_layers > T2_MAX_LAYERS) return TSM_ERR_INVALID;
    if (!dense) {
        if (S < 8 || S > T2_ROWS || (S & (S - 1)) != 0) return TSM_ERR_INVALID;  // whole centres per tile, SC in {8,16,32}
        if (centres >= 0x7fffffffLL) return TSM_ERR_INVALID;                       // 32-bit centre arithmetic
    } else if (S != 1 || a.m != a.n) {
        return TSM_ERR_INVALID;
    }
    Tc2Plan pl;
    pl.nl = a.num_layers;
    pl.eb = eb;
    pl.cl = cl;
    if (!dense) {
        pl.cp = round_up2(a.c_feat, epc);
        pl.xyz_chunk = a.use_xyz ? (pl.cp / epc) : -1;
        pl.K[0] = round_up2(pl.cp + (a.use_xyz ? epc : 0), ks);
    } else {
        pl.cp = 0;
        pl.xyz_chunk = -1;
        pl.K[0] = round_up2(a.c_feat + a.c1, ks);
    }
    int off = 0, kmax = pl.K[0], nmid = 0;
    int nfull_prev = 0;
    for (int l = 0; l < pl.nl; ++l) {
        const bool last = l + 1 == pl.nl;
        const int nfull = round_up2(a.ch[l + 1], last ? T2_ROWS : 16);  // all output channels, padded
        if (nfull > 256) return TSM_ERR_INVALID;
        // a pair splits every layer's output channels in halves: 16-channel granularity, one 128-block each at the end
        if (cl == 2 && (last ? nfull != 2 * T2_ROWS : nfull % 32 != 0)) return TSM_ERR_INVALID;
        pl.Npad[l] = nfull / cl;
        if (l > 0) pl.K[l] = nfull_prev;
        nfull_prev = nfull;
        kmax = pl.K[l] > kmax ? pl.K[l] : kmax;
        if (!last) nmid = pl.Npad[l] > nmid ? pl.Npad[l] : nmid;
        pl.w_off[l] = off;
        off += pl.Npad[l] * (pl.K[l] + (last ? 0 : ks)) * eb;
    }
    for (int l = pl.nl; l < T2_MAX_LAYERS; ++l) pl.K[l] = pl.Npad[l] = pl.w_off[l] = 0;
    if (kmax > 512) return TSM_ERR_INVALID;
    pl.mb = pl.Npad[pl.nl - 1] / T2_ROWS;
    pl.whole_tiles = (!dense && (a.m % (T2_ROWS / S)) == 0) ? 1 : 0;
    pl.b_off = off;
    off += pl.Npad[pl.nl - 1] * 4;
    pl.ones_off = off;  // offsets so far are multiples of 32; descriptors address 16-byte units
    off += 2 * T2_ROWS * 16;
    pl.packed_bytes = off;  // multiple of 32
    off = round_up2(off, 128);
    pl.a_off = off;
    pl.a_bytes = round_up2(T2_ROWS * kmax * eb, 128);
    const bool xch = !dense && S == T2_ROWS;
    auto smem_for = [&](int groups) { return off + groups * pl.a_bytes + (xch ? groups * 2 * T2_ROWS * 4 : 0); };
    if (smem_for(1) > 227 * 1024 - 64) return TSM_ERR_INVALID;
    const int need_cols = nmid > pl.mb * T2_ROWS ? nmid : pl.mb * T2_ROWS;
    pl.grp_cols = 32;
    while (pl.grp_cols < need_cols) pl.grp_cols <<= 1;
    if (pl.grp_cols > 512) return TSM_ERR_INVALID;
    // two tile groups per CTA when the weights allow only one CTA per SM but a second operand buffer still fits
    int groups = 1;
    if (cl == 1 && (227 * 1024) / (smem_for(1) + 2048) < 2 && smem_for(2) <= 227 * 1024 - 64 && 2 * pl.grp_cols <= 512 &&
        !tsm_knob(KNOB_MLP_ONE_GROUP))
        groups = 2;
    pl.tmem_cols = pl.grp_cols * groups;
    pl.x_off = xch ? off + groups * pl.a_bytes : -1;
    pl.smem_bytes = smem_for(groups);
    pl.cls_off = -1;  // set by the launcher when width-class tiles fit behind the plan (tc2_classed)
    pl.ncls = 0;
    *out = pl;
    *groups_out = groups;
    return TSM_OK;
}

// One CTA per tile where the operands fit its shared memory; tf32 SA scales that do not (4-byte weights) go to a cluster
// pair with half of every layer's output channels per CTA.
static int tc2_plan(const tsm::SaMlpArgs& a, long long centres, int dense, int eb, tsm::Tc2Plan* out, int* groups_out) {
    int rc = tc2_plan_cl(a, centres, dense, eb, 1, out, groups_out);
    if (rc == TSM_ERR_INVALID && eb == 4 && !dense) rc = tc2_plan_cl(a, centres, dense, eb, 2, out, groups_out);
    return rc;
}

// Width-class tiles for an SA scale: the 64-byte tile table goes behind the plan's shared memory (the plan itself --
// weight image, groups, cluster pair -- stays as for fixed-width tiles, which the call keeps where the table does
// not fit or would cost a resident CTA).  TSMDET_MLP_WIDTH=fixed: always fixed-width tiles; =classes: a call the width
// classes do not take fails (TSM_ERR_INVALID) instead -- tests use it to know which path they compared.
static bool tc2_classed(tsm::Tc2Plan& pl, int nsample) {
    using namespace tsm;
    const int bytes = 2 * T2_MAX_CLS * 4;
    if (pl.smem_bytes + bytes > 227 * 1024 - 64) return false;
    if ((227 * 1024) / (pl.smem_bytes + bytes + 2048) < (227 * 1024) / (pl.smem_bytes + 2048)) return false;
    pl.cls_off = pl.smem_bytes;
    pl.smem_bytes += bytes;
    pl.ncls = 32 - __builtin_clz((unsigned)nsample);  // nsample = 2^(ncls - 1)
    return true;
}

// The kernel's weight image (bf16 UMMA core matrices incl. the bias steps, the last fp32 bias, the ones operand) for an
// MLP: *bytes = its size; packed != nullptr: build it there (device memory, >= *bytes).  Callers with constant weights
// build it ONCE and pass it to every call (the packing kernel costs 5-8 us, comparable to a whole SA layer's tensor work).
int tsm_mlp_tc2_pack(const tsm::SaMlpArgs& a, int dense, int eb, unsigned char* packed, long long* bytes, cudaStream_t stream) {
    using namespace tsm;
    Tc2Plan pl;
    int groups = 1;
    int rc = tc2_plan(a, 1, dense, eb, &pl, &groups);
    if (rc != TSM_OK) return rc;
    if (bytes) *bytes = (long long)pl.packed_bytes * pl.cl;
    if (packed) {
        for (int l = 0; l < pl.nl; ++l)
            if (!a.w[l] || !a.bias[l]) return TSM_ERR_INVALID;
        dim3 pgrid(16, (unsigned)pl.nl + 1, (unsigned)pl.cl);
        pack_weights2_kernel<<<pgrid, 256, 0, stream>>>(a, pl, dense, packed);
        TSM_LAUNCH_CHECK();
    }
    return TSM_OK;
}

// dense != 0: point-wise MLP over (B, c_feat + c1, n) (a.features / a.src1), a.m == a.n, a.s == 1, no idx.
// prepacked: the image built by tsm_mlp_tc2_pack for the same shapes (nullptr: packed here, per call).
// eb: 2 = bf16 operands, 4 = tf32 operands (a.feat_t / a.out_t rows and the weight image are of that type).
int tsm_mlp_tc2(const tsm::SaMlpArgs& a, int b, int dense, int eb, cudaStream_t stream, const unsigned char* prepacked) {
    using namespace tsm;
    const int S = a.s;
    Tc2Plan pl;
    int groups = 1;
    {
        const int rc = tc2_plan(a, (long long)b * a.m, dense, eb, &pl, &groups);
        if (rc != TSM_OK) return rc;
    }
    const int epc = 16 / eb;
    // feature rows: <= 4 channels are read straight from the (B,C,N) fp32 planes by the gather; wider inputs go
    // through a bf16 (B,N,Cp) transpose so that a gathered row is one contiguous run of 16-byte chunks
    const unsigned char* featT = nullptr;
    if (!dense && a.c_feat > 0 && a.feat_t) {
        featT = (const unsigned char*)a.feat_t;  // rows already in the gather's layout (a previous layer's out_t)
    } else if (!dense && a.c_feat > 4) {
        void* p = nullptr;
        const size_t bytes = (size_t)b * a.n * pl.cp * eb;
        int rc = tsm_scratch_get(1, bytes, stream, &p);
        if (rc != TSM_OK) return rc;
        featT = (const unsigned char*)p;
        dim3 grid((unsigned)divup(a.n, TR_PTS), (unsigned)b);
        const size_t tsm_bytes = (size_t)TR_PTS * (pl.cp + (eb == 2 ? 2 : 1)) * eb;
        if (eb == 2) {
            if (tsm_bytes > 48 * 1024)
                TSM_CUDA_TRY(cudaFuncSetAttribute(transpose2_kernel<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm_bytes));
            transpose2_kernel<__nv_bfloat16><<<grid, 256, tsm_bytes, stream>>>(a.c_feat, pl.cp, a.n, a.features, (__nv_bfloat16*)p);
        } else {
            if (tsm_bytes > 48 * 1024)
                TSM_CUDA_TRY(cudaFuncSetAttribute(transpose2_kernel<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tsm_bytes));
            transpose2_kernel<float><<<grid, 256, tsm_bytes, stream>>>(a.c_feat, pl.cp, a.n, a.features, (float*)p);
        }
        TSM_LAUNCH_CHECK();
    }
    // fixed-width tiles; the grid is sized for them.  (Width classes make up to ncls - 1 more tiles when all classes end
    // in partial tiles -- the persistent loop takes any count.)
    const long long tiles = (a.total_rows + T2_ROWS - 1) / T2_ROWS;
    if (tiles > 0x7fffffffLL) return TSM_ERR_INVALID;
    int* cls = nullptr;
    const char* wk = dense ? nullptr : tsm_knob(KNOB_MLP_WIDTH);
    const bool want_classes = !dense && !(wk && strcmp(wk, "fixed") == 0);
    if (want_classes && !tc2_classed(pl, S) && wk && strcmp(wk, "classes") == 0) return TSM_ERR_INVALID;
    if (pl.cls_off >= 0) {
        const long long centres = (long long)b * a.m;
        void* p = nullptr;
        int rc = tsm_scratch_get(15, (T2_CLS_LIST + (size_t)pl.ncls * centres) * sizeof(int), stream, &p);
        if (rc != TSM_OK) return rc;
        cls = static_cast<int*>(p);
        TSM_CUDA_TRY(cudaMemsetAsync(cls, 0, T2_CLS_LIST * sizeof(int), stream));
        sa_width_classify_kernel<<<(unsigned)divup((int)centres, 256), 256, 0, stream>>>(a.idx, a.idx_cnt, (int)centres, S, cls);
        TSM_LAUNCH_CHECK();
    }
    using Kern = void (*)(const SaMlpArgs, const Tc2Plan, const unsigned char*, const unsigned char*, const int, const int*);
    Kern kern = nullptr;
    // threads per tile row (see the kernel's comment), TSMDET_MLP_NH=1|2 overrides (bf16 SA scales only)
    int nh = dense ? 2 : 1;  // measured (B200, config 2 / config 4): SA L1/L2/L3 48/36/50 us vs 74/48/60, FP MLP 285 vs 233 us
    if (const char* e = tsm_knob(KNOB_MLP_NH)) nh = (atoi(e) == 2 && (eb == 2 || dense)) ? 2 : (dense && eb == 4 ? 2 : 1);
    const int sc = S < 32 ? S : 32;
    const int fchunks = (!dense && featT) ? (pl.cp / epc + pl.cl - 1) / pl.cl : 0;  // register-prefetched chunks per CTA
    const int pf = fchunks == 0 ? 0 : (fchunks <= 4 ? 4 : (fchunks <= 16 ? 16 : 0));
    // MINB: one-group CTAs of 128 threads with narrow rows fit 4 per SM in <= 128 registers; 256-thread ones 2
#define TC2_PICK(G, P, H, B, E)                                                                                       \
    (sc == 32 ? mlp_tc2_kernel<G, 32, false, P, H, B, E>                                                              \
              : (sc == 16 ? mlp_tc2_kernel<G, 16, false, P, H, B, E> : mlp_tc2_kernel<G, 8, false, P, H, B, E>))
#define TC2_PICK_PF(G, H, B16, B4, E) (pf == 16 ? TC2_PICK(G, 16, H, B16, E) : (pf == 4 ? TC2_PICK(G, 4, H, B4, E) : TC2_PICK(G, 0, H, B4, E)))
    if (eb == 2) {
        if (dense) {
            if (nh == 2) kern = groups == 2 ? mlp_tc2_kernel<2, 32, true, 0, 2, 1, 2> : mlp_tc2_kernel<1, 32, true, 0, 2, 2, 2>;
            else kern = groups == 2 ? mlp_tc2_kernel<2, 32, true, 0, 1, 1, 2> : mlp_tc2_kernel<1, 32, true, 0, 1, 2, 2>;
        } else if (nh == 2) {
            kern = groups == 2 ? TC2_PICK_PF(2, 2, 1, 1, 2) : TC2_PICK_PF(1, 2, 2, 2, 2);
        } else {
            kern = groups == 2 ? TC2_PICK_PF(2, 1, 1, 1, 2) : TC2_PICK_PF(1, 1, 1, 4, 2);
        }
    } else {  // tf32: one thread per row for SA scales, two for dense MLPs
        if (dense) {
            kern = groups == 2 ? mlp_tc2_kernel<2, 32, true, 0, 2, 1, 4> : mlp_tc2_kernel<1, 32, true, 0, 2, 2, 4>;
        } else if (pl.cl == 2) {
#define TC2_PICK2(P) (sc == 32 ? mlp_tc2_kernel<1, 32, false, P, 1, 1, 4, 2> : (sc == 16 ? mlp_tc2_kernel<1, 16, false, P, 1, 1, 4, 2> : mlp_tc2_kernel<1, 8, false, P, 1, 1, 4, 2>))
            kern = pf == 16 ? TC2_PICK2(16) : (pf == 4 ? TC2_PICK2(4) : TC2_PICK2(0));
#undef TC2_PICK2
        } else {
            kern = groups == 2 ? TC2_PICK_PF(2, 1, 1, 1, 4) : TC2_PICK_PF(1, 1, 1, 4, 4);
        }
    }
#undef TC2_PICK_PF
#undef TC2_PICK
    const int gthreads = 128 * nh;
    TSM_CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, pl.smem_bytes));
    // resident CTAs per SM: what shared memory, registers (a grid of more CTAs than are resident runs a second,
    // partial wave) and the 512 TMEM columns allow
    int occ = (227 * 1024) / (pl.smem_bytes + 2048);
    {
        cudaFuncAttributes fa;
        cudaError_t e = cudaFuncGetAttributes(&fa, kern);
        if (e == cudaSuccess && fa.numRegs > 0) {
            const int regs_cta = ((fa.numRegs + 7) / 8 * 8) * gthreads * groups;
            const int occ_regs = 65536 / regs_cta;
            if (occ > occ_regs) occ = occ_regs;
        } else {
            cudaGetLastError();
            if (occ > 2) occ = 2;
        }
    }
    const int tmem_occ = 512 / pl.tmem_cols;
    if (occ > tmem_occ) occ = tmem_occ;
    if (occ < 1) occ = 1;
    if (const char* e = tsm_knob(KNOB_MLP_OCC)) occ = atoi(e) > 0 && atoi(e) < occ ? atoi(e) : occ;
    long long grid = (long long)tsm_num_sms() * occ;
    if (grid * groups > tiles) grid = (tiles + groups - 1) / groups;
    if (pl.cl == 2) {  // pairs: both CTAs of a cluster walk the same tiles
        long long clusters = (long long)(tsm_num_sms() / 2) * occ;
        if (clusters > tiles) clusters = tiles;
        grid = 2 * clusters;
    }
    SaMlpArgs args = a;
    args.status = tsm_status_word(stream);
    const unsigned char* packed = prepacked;
    if (!packed) {
        void* p = nullptr;
        int rc = tsm_scratch_get(2, (size_t)pl.packed_bytes * pl.cl, stream, &p);
        if (rc != TSM_OK) return rc;
        dim3 pgrid(16, (unsigned)pl.nl + 1, (unsigned)pl.cl);
        pack_weights2_kernel<<<pgrid, 256, 0, stream>>>(args, pl, dense, (unsigned char*)p);
        TSM_LAUNCH_CHECK();
        packed = (const unsigned char*)p;
    }
    if (pl.cl == 2) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)grid);
        cfg.blockDim = dim3((unsigned)(gthreads * groups));
        cfg.dynamicSmemBytes = (size_t)pl.smem_bytes;
        cfg.stream = stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2;
        attr[0].val.clusterDim.y = 1;
        attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
        const int ntiles = (int)tiles;
        TSM_CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, args, pl, featT, packed, ntiles, (const int*)cls));
    } else {
        kern<<<(unsigned)grid, gthreads * groups, pl.smem_bytes, stream>>>(args, pl, featT, packed, (int)tiles, cls);
    }
    TSM_LAUNCH_CHECK();
    return TSM_OK;
}
