// Error reporting and device-attribute cache for the C ABI.
#include <stdarg.h>
#include <stdlib.h>

#include "mf_common.cuh"

static thread_local char g_err[512] = "";

void mf_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

MF_API const char* mf_last_error(void) { return g_err; }
MF_API int mf_abi_version(void) { return MF_ABI_VERSION; }

int mf_sm_count_cached() {
    static int cached[64] = {0};
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
    if (cached[dev] == 0) {
        int n = 0;
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        cached[dev] = n;
    }
    return cached[dev];
}

// SMs the producer / consumer forward kernel leaves free (its persistent CTAs fill an SM completely): lets a small collective
// kernel issued on another stream -- the data-parallel mapper's 16-byte count all-reduce -- run beside it instead of behind it.
static int g_sm_reserve = 0;
int mf_sm_reserve() { return g_sm_reserve; }
MF_API int mf_set_sm_reserve(int n) {
    MF_CHECK_ARG(n >= 0 && n < 32);
    g_sm_reserve = n;
    return MF_OK;
}

MF_API int mf_device_sm_count(void) {
    int dev = 0, n = 0;
    MF_CUDA(cudaGetDevice(&dev));
    MF_CUDA(cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev));
    return n;
}

// ---- decoder implementation switch + tensor-core error flag ------------------------------------
static int g_decoder_impl = 0;
int mf_decoder_impl() { return g_decoder_impl; }

MF_API int mf_set_decoder_impl(int impl) {
    // 0: tcgen05 (producer / consumer forward), 1: fp32 CUDA cores; A/B comparisons of the tcgen05 forward:
    // 2: single pipeline, 3: dual pipeline
    MF_CHECK_ARG(impl >= 0 && impl <= 3);
    g_decoder_impl = impl;
    return MF_OK;
}
MF_API int mf_get_decoder_impl(void) { return g_decoder_impl; }

// A/B switch of the tensor-core backward: 0 three-role kernel (field_tc_bwd2.cuh, default), 1 single-role kernel
// (field_tc_bwd.cuh), 2 three-role kernel without the warp-aggregated scatter, 3 four-role kernel (field_tc_bwd3.cuh: correct,
// measured slower).
static int g_bwd_impl = 0;
int mf_bwd_impl() { return g_bwd_impl; }
MF_API int mf_set_bwd_impl(int impl) {
    MF_CHECK_ARG(impl >= 0 && impl <= 3);
    g_bwd_impl = impl;
    return MF_OK;
}

static int* g_tile_ctr[64] = {nullptr};
static unsigned g_tile_next[64] = {0};
static int g_dynamic_tiles = 1;
constexpr int TILE_CTR_RING = 256;
int* mf_tile_counter() {
    if (!g_dynamic_tiles) return nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!g_tile_ctr[dev]) {
        if (cudaMalloc(&g_tile_ctr[dev], TILE_CTR_RING * 2 * sizeof(int)) != cudaSuccess) return nullptr;
        cudaMemset(g_tile_ctr[dev], 0, TILE_CTR_RING * 2 * sizeof(int));
    }
    return g_tile_ctr[dev] + 2 * (g_tile_next[dev]++ % TILE_CTR_RING);
}
// A/B switch: 1 (default) = tiles of the producer / consumer forward kernel are drawn from a global counter, 0 = static striding.
MF_API int mf_set_dynamic_tiles(int on) {
    g_dynamic_tiles = on ? 1 : 0;
    return MF_OK;
}

// Programmatic dependent launch of the map step's kernels (mf_launch, mf_common.cuh): on unless MF_NO_PDL=1; mf_set_pdl switches
// it at run time (A/B of both launch modes in one process).
static int g_pdl = -1;
bool mf_pdl_enabled() {
    if (g_pdl < 0) {
        const char* e = getenv("MF_NO_PDL");
        g_pdl = (e && e[0] && strcmp(e, "0") != 0) ? 0 : 1;
    }
    return g_pdl != 0;
}
MF_API int mf_set_pdl(int on) {
    g_pdl = on ? 1 : 0;
    return MF_OK;
}
MF_API int mf_get_pdl(void) { return mf_pdl_enabled() ? 1 : 0; }

// Deterministic mode (det_kernels.cu): off unless MF_DETERMINISTIC=1; mf_set_deterministic switches it at run time.
static int g_det = -1;
bool mf_deterministic() {
    if (g_det < 0) {
        const char* e = getenv("MF_DETERMINISTIC");
        g_det = (e && e[0] && strcmp(e, "0") != 0) ? 1 : 0;
    }
    return g_det != 0;
}
MF_API int mf_set_deterministic(int on) {
    g_det = on ? 1 : 0;
    return MF_OK;
}
MF_API int mf_get_deterministic(void) { return mf_deterministic() ? 1 : 0; }

static int* g_tc_err[64] = {nullptr};
int* mf_tc_error_flag() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!g_tc_err[dev]) {
        if (cudaMalloc(&g_tc_err[dev], sizeof(int)) != cudaSuccess) return nullptr;
        cudaMemset(g_tc_err[dev], 0, sizeof(int));
    }
    return g_tc_err[dev];
}

// Returns 1 if any tensor-core kernel on the current device reported an MMA completion timeout since the
// last call (and clears the flag).  Synchronises the device: diagnostics only.
MF_API int mf_tc_check_error(void) {
    int* p = mf_tc_error_flag();
    if (!p) return MF_ERR_CUDA;
    int v = 0;
    MF_CUDA(cudaMemcpy(&v, p, sizeof(int), cudaMemcpyDeviceToHost));
    if (v) MF_CUDA(cudaMemset(p, 0, sizeof(int)));
    return v;
}

// ---- in-kernel phase profiling (diagnostics) -----------------------------------------------------
static long long* g_prof[64] = {nullptr};
static int g_prof_on = 0;
long long* mf_tc_profile_buffer() {
    if (!g_prof_on) return nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!g_prof[dev]) {
        if (cudaMalloc(&g_prof[dev], MF_PROF_SLOTS * sizeof(long long)) != cudaSuccess) return nullptr;
        cudaMemset(g_prof[dev], 0, MF_PROF_SLOTS * sizeof(long long));
    }
    return g_prof[dev];
}
// Enable (on != 0) / disable the clock stamps the tensor-core backward kernel records for its second tile on
// CTA 0; out_host (64 int64, may be NULL) receives the last recorded stamps.  Synchronises the device.
MF_API int mf_debug_profile(int on, long long* out_host) {
    g_prof_on = on ? 1 : 0;
    if (out_host) {
        int dev = 0;
        MF_CUDA(cudaGetDevice(&dev));
        if (g_prof[dev]) MF_CUDA(cudaMemcpy(out_host, g_prof[dev], 64 * sizeof(long long), cudaMemcpyDeviceToHost));
        else memset(out_host, 0, 64 * sizeof(long long));
    }
    return MF_OK;
}

// All MF_PROF_SLOTS stamps: [0, 64) as mf_debug_profile; [64 + 2 b, +1] = globaltimer (ns) at the start / end of CTA b of the last
// profiled field_fwd_tc3_kernel, [576 + 2 b, +1] the same for field_bwd_tc2_kernel (b < 256).
MF_API int mf_debug_profile_all(long long* out_host, int n) {
    MF_CHECK_ARG(out_host && n >= 0 && n <= MF_PROF_SLOTS);
    int dev = 0;
    MF_CUDA(cudaGetDevice(&dev));
    if (g_prof[dev]) MF_CUDA(cudaMemcpy(out_host, g_prof[dev], (size_t)n * sizeof(long long), cudaMemcpyDeviceToHost));
    else memset(out_host, 0, (size_t)n * sizeof(long long));
    return MF_OK;
}

// ---- per-kernel device timing (diagnostics; bench.py's roofline line) ----------------------------
// When enabled, the launchers of the dominant kernels bracket the kernel launch itself with a CUDA event pair on the
// launching stream (slot 0: field forward, 1: field backward, 2: RandomOptimizer field query, 3: joint-query field query).
static int g_ktimer_on = 0;
static cudaEvent_t g_kev[64][MF_KTIMER_SLOTS][2];
static bool g_kev_init[64] = {false};
static cudaEvent_t* ktimer_events(int slot) {
    if (!g_ktimer_on || slot < 0 || slot >= MF_KTIMER_SLOTS) return nullptr;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return nullptr;
    if (!g_kev_init[dev]) {
        for (int s = 0; s < MF_KTIMER_SLOTS; ++s)
            for (int k = 0; k < 2; ++k)
                if (cudaEventCreate(&g_kev[dev][s][k]) != cudaSuccess) return nullptr;
        g_kev_init[dev] = true;
    }
    return g_kev[dev][slot];
}
void mf_ktimer_begin(int slot, cudaStream_t st) { if (cudaEvent_t* e = ktimer_events(slot)) cudaEventRecord(e[0], st); }
void mf_ktimer_end(int slot, cudaStream_t st) { if (cudaEvent_t* e = ktimer_events(slot)) cudaEventRecord(e[1], st); }

MF_API int mf_debug_kernel_timer(int on) { g_ktimer_on = on ? 1 : 0; return MF_OK; }
// Duration (ms) of the last launch bracketed in `slot`.  Waits for that launch to finish.
MF_API int mf_debug_kernel_ms(int slot, float* ms) {
    MF_CHECK_ARG(ms != nullptr && slot >= 0 && slot < MF_KTIMER_SLOTS);
    cudaEvent_t* e = ktimer_events(slot);
    if (!e) { mf_set_error("mf_debug_kernel_ms: the kernel timer is off"); return MF_ERR_INVALID; }
    MF_CUDA(cudaEventSynchronize(e[1]));
    MF_CUDA(cudaEventElapsedTime(ms, e[0], e[1]));
    return MF_OK;
}
