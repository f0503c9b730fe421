// runtime.cu -- process-wide host helpers of the C-ABI library.
#include <mutex>
#include <string>
#include <vector>
#include <stdlib.h>

#include "common.cuh"

static std::mutex g_mu;
static int g_sms[64];
static int* g_status[64];       // device-side address of the status word (host-mapped pinned memory)
static int* g_status_host[64];  // the same word as the host sees it

// ---- TSMDET_* tuning knobs: read from the environment ONCE (first use) into a table, so no launch path calls
// getenv(); tsmdet_reload_options() re-reads them (tests and tuning scripts flip knobs between calls).
static const char* const kKnobNames[KNOB_COUNT] = {
    "TSMDET_BQ_ALGO",       "TSMDET_FPS_CLUSTER",  "TSMDET_FPS_THREADS",     "TSMDET_FPS_ALGO",   "TSMDET_FPSB_T",
    "TSMDET_FPSB_P",        "TSMDET_FPSB_K",       "TSMDET_GROUP_SLAB_KB",   "TSMDET_GROUP_WAVES", "TSMDET_GROUP_DIRECT",
    "TSMDET_NN_ALGO",       "TSMDET_NMS_CTAS_PER_SM", "TSMDET_NMS_ALGO",     "TSMDET_MLP_ONE_GROUP", "TSMDET_MLP_OCC",
    "TSMDET_MLP_V1",        "TSMDET_FPSC_K",       "TSMDET_VOXEL_ALGO",      "TSMDET_MLP_NH",     "TSMDET_MLP_WIDTH",
};
static std::string g_knob_val[KNOB_COUNT];
static bool g_knob_set[KNOB_COUNT];
static std::once_flag g_knob_once;
static std::mutex g_knob_mu;

static void knobs_load() {
    std::lock_guard<std::mutex> lk(g_knob_mu);
    for (int i = 0; i < KNOB_COUNT; ++i) {
        const char* e = getenv(kKnobNames[i]);
        g_knob_set[i] = e != nullptr;
        g_knob_val[i] = e ? e : "";
    }
}

const char* tsm_knob(int id) {
    if (id < 0 || id >= KNOB_COUNT) return nullptr;
    std::call_once(g_knob_once, knobs_load);
    return g_knob_set[id] ? g_knob_val[id].c_str() : nullptr;
}

int tsm_num_sms() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    std::lock_guard<std::mutex> lk(g_mu);
    if (g_sms[dev] == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) v = 148;
        g_sms[dev] = v;
    }
    return g_sms[dev];
}

// One zero-initialised int per device in MAPPED PINNED HOST memory: kernels with in-kernel waits record a
// watchdog code here, so the host can still read it after a kernel fault has poisoned the context (a word in
// cudaMalloc memory cannot be copied back once the context carries a sticky error).
int* tsm_status_word(cudaStream_t) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    std::lock_guard<std::mutex> lk(g_mu);
    if (!g_status[dev]) {
        int* h = nullptr;
        int* d = nullptr;
        if (cudaHostAlloc((void**)&h, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable) != cudaSuccess) {
            cudaGetLastError();
            return nullptr;
        }
        *h = 0;
        if (cudaHostGetDevicePointer((void**)&d, h, 0) != cudaSuccess) {
            cudaGetLastError();
            cudaFreeHost(h);
            return nullptr;
        }
        g_status_host[dev] = h;
        g_status[dev] = d;
    }
    return g_status[dev];
}

struct Retired {
    void* p;
    size_t bytes;
    int dev;
};
static std::vector<Retired> g_retired;  // outgrown / evicted buffers: freed by tsmdet_scratch_trim()
static size_t g_retired_bytes = 0;

struct Scratch {
    void* p = nullptr;
    size_t cap = 0;
    int dev = -1;
    cudaStream_t stream = nullptr;
    int tag = 0;
    unsigned long long tick = 0;
};
// Grow-only device scratch, one buffer per (device, stream, user tag) so that calls on
// different streams never share a buffer; stream-ordered (cudaMallocAsync), so repeated
// NMS calls allocate nothing.
constexpr int kScratchSlots = 256;  // (device, stream, tag) keys: 8 pipeline lanes x 3 streams x 6 tags and room to spare
static Scratch g_scratch[kScratchSlots];
static unsigned long long g_tick = 0;
static std::mutex g_scratch_mu;

int tsm_scratch_get(int tag, size_t bytes, cudaStream_t s, void** out) {
    int dev = 0;
    TSM_CUDA_TRY(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    Scratch* sc = nullptr;
    for (auto& e : g_scratch)
        if (e.p && e.dev == dev && e.stream == s && e.tag == tag) sc = &e;
    if (!sc) {  // empty slot, else evict the least recently used one
        for (auto& e : g_scratch)
            if (!e.p && !sc) sc = &e;
        if (!sc) {
            sc = &g_scratch[0];
            for (auto& e : g_scratch)
                if (e.tick < sc->tick) sc = &e;
            if (sc->p) {  // retired (see below)
                g_retired.push_back({sc->p, sc->cap, sc->dev});
                g_retired_bytes += sc->cap;
            }
            sc->p = nullptr;
            sc->cap = 0;
        }
        sc->dev = dev;
        sc->stream = s;
        sc->tag = tag;
    }
    sc->tick = ++g_tick;
    if (sc->cap < bytes) {
        // The outgrown buffer is RETIRED, not freed here: a captured CUDA graph may still hold its address.
        // Retired buffers are kept on a list and released by tsmdet_scratch_trim() (call it when no captured
        // graph that ran through this library is alive any more, e.g. after re-capturing for new shapes).
        if (sc->p) {
            g_retired.push_back({sc->p, sc->cap, sc->dev});
            g_retired_bytes += sc->cap;
        }
        sc->p = nullptr;
        sc->cap = 0;
        const size_t want = bytes + bytes / 4;
        TSM_CUDA_TRY(cudaMallocAsync(&sc->p, want, s));
        sc->cap = want;
    }
    *out = sc->p;
    return TSM_OK;
}


extern "C" {

const char* tsmdet_version() { return "tsmdet_b200 0.1 (sm_100a)"; }

// Human-readable text for a status returned by any tsmdet_* entry point.
const char* tsmdet_error_string(int code) {
    if (code == TSM_OK) return "ok";
    if (code == TSM_ERR_INVALID) return "tsmdet: invalid argument or unsupported size";
    if (code == TSM_ERR_WATCHDOG) return "tsmdet: in-kernel wait timed out";
    return cudaGetErrorString((cudaError_t)code);
}

// Reads (and clears) the watchdog status word of the current device; 0 = clean.  The word lives in mapped pinned
// host memory, so this needs no CUDA call and still works after a kernel fault.
int tsmdet_read_status() {
    if (!tsm_status_word(nullptr)) return 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
    volatile int* h = g_status_host[dev];
    if (!h) return 0;
    const int v = *h;
    if (v) *h = 0;
    return v;
}

// Re-reads the TSMDET_* tuning knobs from the environment (they are otherwise read once, at first use).
int tsmdet_reload_options() {
    std::call_once(g_knob_once, [] {});
    knobs_load();
    return TSM_OK;
}

// Scratch-pool accounting: bytes held by live (device, stream, tag) buffers and by retired ones.
int tsmdet_scratch_stats(long long* live_bytes, long long* retired_bytes) {
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    long long live = 0;
    for (auto& e : g_scratch)
        if (e.p) live += (long long)e.cap;
    if (live_bytes) *live_bytes = live;
    if (retired_bytes) *retired_bytes = (long long)g_retired_bytes;
    return TSM_OK;
}

// Frees every retired scratch buffer (device-synchronising).  The caller guarantees that no captured CUDA graph
// recorded through this library before the call is replayed afterwards.
int tsmdet_scratch_trim() {
    std::lock_guard<std::mutex> lk(g_scratch_mu);
    int cur = 0;
    TSM_CUDA_TRY(cudaGetDevice(&cur));
    for (auto& r : g_retired) {
        cudaSetDevice(r.dev);
        cudaDeviceSynchronize();
        cudaFree(r.p);
    }
    cudaSetDevice(cur);
    g_retired.clear();
    g_retired_bytes = 0;
    return TSM_OK;
}

}  // extern "C"
