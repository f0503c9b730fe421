// common.cuh -- shared device/host helpers for the sm_100a kernels of this library.
//
// Numerics contract (SURVEY.md section 9, verified against the SASS of the
// reference build, oracle/_ref): every squared distance on this path is
//     d2 = fma(dz, dz, fma(dx, dx, dy * dy)),   dx = x2 - x1 rounded to f32 first
// We spell it with explicit round-to-nearest intrinsics so the result never
// depends on the compiler's contraction choices.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#define TSM_OK 0
#define TSM_ERR_INVALID 1000001   // bad argument (shape / unsupported size)
#define TSM_ERR_WATCHDOG 1000002  // an in-kernel wait timed out (reported via status word)

#define TSM_CUDA_TRY(expr)                          \
    do {                                            \
        cudaError_t _e = (expr);                    \
        if (_e != cudaSuccess) return (int)_e;      \
    } while (0)

#define TSM_LAUNCH_CHECK()                          \
    do {                                            \
        cudaError_t _e = cudaGetLastError();        \
        if (_e != cudaSuccess) return (int)_e;      \
    } while (0)

namespace tsm {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ float sqdist3(float x1, float y1, float z1, float x2, float y2, float z2) {
    const float dx = __fsub_rn(x2, x1);
    const float dy = __fsub_rn(y2, y1);
    const float dz = __fsub_rn(z2, z1);
    return __fmaf_rn(dz, dz, __fmaf_rn(dx, dx, __fmul_rn(dy, dy)));
}

// The same squared distance for TWO points at once with sm_100's packed fp32 instructions (FADD2 / FMUL2 / FFMA2: each
// component is the IEEE round-to-nearest operation, so both results are bit-identical to sqdist3): six instructions per
// pair instead of twelve.  n1 = the NEGATED pick coordinate in both halves (x2 - x1 == x2 + (-x1) exactly).
__device__ __forceinline__ unsigned long long f2_pack(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ float2 f2_unpack(unsigned long long v) {
    float2 r;
    asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(v));
    return r;
}
__device__ __forceinline__ float2 sqdist3_x2(unsigned long long nx1, unsigned long long ny1, unsigned long long nz1, float xa, float xb,
                                             float ya, float yb, float za, float zb) {
    unsigned long long dx, dy, dz, m;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(dx) : "l"(f2_pack(xa, xb)), "l"(nx1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(dy) : "l"(f2_pack(ya, yb)), "l"(ny1));
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(dz) : "l"(f2_pack(za, zb)), "l"(nz1));
    asm("mul.rn.f32x2 %0, %1, %1;" : "=l"(m) : "l"(dy));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(m) : "l"(dx), "l"(m));
    asm("fma.rn.f32x2 %0, %1, %1, %2;" : "=l"(m) : "l"(dz), "l"(m));
    return f2_unpack(m);
}

// Order-preserving map float -> uint32 (handles negatives; -0.0 must be
// canonicalised to +0.0 by the caller if ties with +0.0 matter).
__device__ __forceinline__ uint32_t f32_ordered(float v) {
    const uint32_t b = __float_as_uint(v);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return (uint32_t)__cvta_generic_to_shared(p);
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}

__device__ __forceinline__ uint32_t cluster_nctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
    return r;
}

__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}

// Map a local shared-memory address to the same offset in CTA `rank` of the cluster.
__device__ __forceinline__ uint32_t mapa_u32(uint32_t local_addr, uint32_t rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(rank));
    return r;
}

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}

__device__ __forceinline__ void mbar_fence_init_cluster() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}

__device__ __forceinline__ bool mbar_try_wait_cluster(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}

__device__ __forceinline__ bool mbar_try_wait_cta(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}

// non-blocking probe of a phase (test_wait returns at once; try_wait may suspend the thread)
__device__ __forceinline__ bool mbar_test_wait_cta(uint32_t bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}

// Remote (DSMEM) store that completes `bytes` on the destination CTA's mbarrier.
__device__ __forceinline__ void st_async_v4(uint32_t raddr, uint32_t rbar, uint32_t a, uint32_t b, uint32_t c,
                                            uint32_t d) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                     raddr),
                 "r"(a), "r"(b), "r"(c), "r"(d), "r"(rbar)
                 : "memory");
}

__device__ __forceinline__ void st_async_b32(uint32_t raddr, uint32_t rbar, uint32_t a) {
    asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.b32 [%0], %1, [%2];" ::"r"(raddr),
                 "r"(a), "r"(rbar)
                 : "memory");
}

// 1-D bulk copy global -> shared (TMA engine, SASS: UBLKCP), completing on an mbarrier.
__device__ __forceinline__ void bulk_g2s(uint32_t dst_smem, const void* src_gmem, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     dst_smem),
                 "l"(src_gmem), "r"(bytes), "r"(bar)
                 : "memory");
}

// Watchdog for every INTRA-GPU in-kernel wait (mbarrier phases of one kernel): a mis-programmed barrier must
// end the kernel (trap) rather than hang the GPU.  The status word is host-mapped, so the code survives the
// trap.  (Waits on OTHER ranks -- peer_put.cu -- never trap: they record the code and return.)
__device__ __forceinline__ void watchdog_trip(int* status, int code) {
    if (status) *reinterpret_cast<volatile int*>(status) = code;
    __threadfence_system();
    __trap();
}

__host__ __device__ __forceinline__ int divup(int a, int b) { return (a + b - 1) / b; }

}  // namespace tsm

// Host-side: number of SMs of the current device (cached).
int tsm_num_sms();
int* tsm_status_word(cudaStream_t stream);  // device address of a host-mapped int, zero-initialised, one per device

// TSMDET_* tuning knobs, captured from the environment once (runtime.cu); nullptr = unset.
enum TsmKnob {
    KNOB_BQ_ALGO, KNOB_FPS_CLUSTER, KNOB_FPS_THREADS, KNOB_FPS_ALGO, KNOB_FPSB_T,
    KNOB_FPSB_P, KNOB_FPSB_K, KNOB_GROUP_SLAB_KB, KNOB_GROUP_WAVES, KNOB_GROUP_DIRECT,
    KNOB_NN_ALGO, KNOB_NMS_CTAS_PER_SM, KNOB_NMS_ALGO, KNOB_MLP_ONE_GROUP, KNOB_MLP_OCC,
    KNOB_MLP_V1, KNOB_FPSC_K, KNOB_VOXEL_ALGO, KNOB_MLP_NH, KNOB_MLP_WIDTH,
    KNOB_COUNT
};
const char* tsm_knob(int id);
// Stream-ordered grow-only scratch, keyed by (device, stream, tag): tag 0 = IoU/NMS, 1 = SA MLP.
int tsm_scratch_get(int tag, size_t bytes, cudaStream_t stream, void** out);
