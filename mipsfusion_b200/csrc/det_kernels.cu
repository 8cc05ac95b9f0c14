// Deterministic mode: an order-independent hash-grid gradient by pre-rounded fixed-point accumulation (the ReproBLAS idea).
//
// For every gradient float e of the table, with contributions c = __fmul_rn(w, dy) (w the trilinear corner weight of
// grid_corners, dy the feature gradient: the same products the atomic scatter adds):
//   pass 1  E[e] = max over its non-zero contributions of the effective binary exponent max(biased exponent, 1) (an integer
//           red.max); non-finite contributions set sticky +Inf / -Inf / NaN flags instead (red.or).
//   pass 2  each contribution is rounded to the integer round(c * 2^s), s = 188 - h - E[e], which puts the largest possible
//           magnitude (< 2^(E - 126)) below bit 62 - h; h = ceil(log2(8 N + 1)) bounds the number of contributions one entry
//           can receive in a launch (8 corners per point and level), so the int64 sum cannot overflow.  Integer addition is
//           associative: the sum depends only on the multiset of contributions, not on their order or timing.
//   finalize a sweep over all gradient floats; where E[e] != 0: grad[e] = __fadd_rn(grad[e], float(acc[e]) * 2^-s) (+Inf / -Inf /
//           NaN when flagged, as fp32 arithmetic would give), and acc and E are reset, so the workspace is all-zero between calls.
//           (A list of touched entries appended by pass 1 was measured instead: its one shared counter serialised pass 1 --
//           874 us per bench step against a sweep that reads the 4-byte exponent words of the whole table once.)
// oracle/det_scatter.py restates the arithmetic in numpy; DESIGN §4 (Deterministic mode) gives the accuracy bound.
#include <mutex>
#include <vector>

#include "grid_encode.cuh"

constexpr uint32_t DET_PINF = 1u << 16, DET_NINF = 1u << 17, DET_NAN = 1u << 18, DET_FLAGS = DET_PINF | DET_NINF | DET_NAN;
constexpr int DET_NT = 256;

// thread per (point, level); returns false for threads without work
__device__ __forceinline__ bool det_point(const FieldDev& f, const float* __restrict__ x, int ldx, const float* __restrict__ dy, int ldy,
                                          const int* __restrict__ count, int64_t n, uint32_t (&idx)[8], float (&w)[8], float2& g,
                                          size_t& base) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int L = f.n_levels;
    if (t >= n * L) return false;
    const int64_t i = t / L; const int l = (int)(t % L);
    if (count && i >= (int64_t)*count) return false;
    g = make_float2(dy[i * ldy + 2 * l], dy[i * ldy + 2 * l + 1]);
    if (g.x == 0.f && g.y == 0.f) return false;
    const float xv[3] = {x[i * ldx], x[i * ldx + 1], x[i * ldx + 2]};
    const LevelInfo li = level_info(f, l);
    grid_corners(xv, li, idx, w);
    base = 2 * (size_t)li.offset;                     // 64-bit flat index, as the atomic scatter's: tables of >= 2^31 entries
    return true;
}

__global__ void __launch_bounds__(DET_NT) det_pass1_kernel(FieldDev f, const float* __restrict__ x, int ldx, const float* __restrict__ dy,
                                                           int ldy, const int* __restrict__ count, int64_t n, uint32_t* __restrict__ expo) {
    mf_pdl_wait(); mf_pdl_trigger();
    uint32_t idx[8]; float w[8]; float2 g; size_t base;
    if (!det_point(f, x, ldx, dy, ldy, count, n, idx, w, g, base)) return;
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float v = __fmul_rn(w[c], k ? g.y : g.x);
            if (v == 0.f) continue;
            const size_t e = base + 2 * (size_t)idx[c] + k;
            const uint32_t b = __float_as_uint(v), be = (b >> 23) & 0xffu;
            if (be == 0xffu) atomicOr(&expo[e], (b & 0x7fffffu) ? DET_NAN : ((b >> 31) ? DET_NINF : DET_PINF));
            else atomicMax(&expo[e], be > 1u ? be : 1u);         // (results unused: reductions)
        }
}

__global__ void __launch_bounds__(DET_NT) det_pass2_kernel(FieldDev f, const float* __restrict__ x, int ldx, const float* __restrict__ dy,
                                                           int ldy, const int* __restrict__ count, int64_t n, int h,
                                                           const uint32_t* __restrict__ expo, unsigned long long* __restrict__ acc) {
    mf_pdl_wait(); mf_pdl_trigger();
    uint32_t idx[8]; float w[8]; float2 g; size_t base;
    if (!det_point(f, x, ldx, dy, ldy, count, n, idx, w, g, base)) return;
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const float v = __fmul_rn(w[c], k ? g.y : g.x);
            if (v == 0.f) continue;
            const size_t e = base + 2 * (size_t)idx[c] + k;
            const uint32_t E = __ldg(&expo[e]);
            if (E & DET_FLAGS) continue;                         // the sum is non-finite: finalize ignores acc
            const int s = 188 - h - (int)E;                      // in [-106, 187]: 2^s is a normal double, v * 2^s exact
            const long long q = __double2ll_rn((double)v * __hiloint2double((s + 1023) << 20, 0));
            atomicAdd(&acc[e], (unsigned long long)q);           // two's complement: the unsigned sum is the signed sum
        }
}

__device__ __forceinline__ void det_finalize_one(int h, uint32_t E, int64_t e, uint32_t* __restrict__ expo, unsigned long long* __restrict__ acc,
                                                 float* __restrict__ grad) {
    float v;
    if (E & DET_FLAGS) {
        v = ((E & DET_NAN) || ((E & DET_PINF) && (E & DET_NINF))) ? __int_as_float(0x7fc00000) : ((E & DET_PINF) ? __int_as_float(0x7f800000)
                                                                                                                   : __int_as_float(0xff800000));
    } else {
        const int s = 188 - h - (int)E;
        // one rounding to fp32 of the integer, then an exact scaling in fp64 and (only for a subnormal result) a second rounding
        v = __double2float_rn((double)__ll2float_rn((long long)acc[e]) * __hiloint2double((1023 - s) << 20, 0));
    }
    grad[e] = __fadd_rn(grad[e], v);
    expo[e] = 0u; acc[e] = 0ull;
}

// four exponent words per thread and step (tables from mf_hashgrid_meta have P % 32 == 0; a ragged tail is handled singly)
__global__ void __launch_bounds__(DET_NT) det_finalize_kernel(int h, int64_t P, uint32_t* __restrict__ expo, unsigned long long* __restrict__ acc,
                                                              float* __restrict__ grad) {
    mf_pdl_wait(); mf_pdl_trigger();
    for (int64_t j = (int64_t)blockIdx.x * DET_NT + threadIdx.x; 4 * j < P; j += (int64_t)gridDim.x * DET_NT) {
        if (4 * j + 4 > P) {
            for (int64_t e = 4 * j; e < P; ++e)
                if (const uint32_t E = expo[e]) det_finalize_one(h, E, e, expo, acc, grad);
            continue;
        }
        const uint4 E = __ldcs(reinterpret_cast<const uint4*>(expo) + j);
        if ((E.x | E.y | E.z | E.w) == 0u) continue;                // untouched
        if (E.x) det_finalize_one(h, E.x, 4 * j, expo, acc, grad);
        if (E.y) det_finalize_one(h, E.y, 4 * j + 1, expo, acc, grad);
        if (E.z) det_finalize_one(h, E.z, 4 * j + 2, expo, acc, grad);
        if (E.w) det_finalize_one(h, E.w, 4 * j + 3, expo, acc, grad);
    }
}

// mf_hashgrid_bwd's input gradient without the table scatter
__global__ void hashgrid_bwd_dx_kernel(FieldDev f, const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx_out,
                                       int64_t N) {
    hashgrid_bwd_body<true, false>(f, x, dy, nullptr, dx_out, N);
}

int mf_det_hashgrid_dx(const FieldDev& f, const float* x, const float* dy, float* dx, int64_t N, cudaStream_t st) {
    hashgrid_bwd_dx_kernel<<<(unsigned)((N * f.n_levels + 255) / 256), 256, 0, st>>>(f, x, dy, dx, N);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Host side: workspaces keyed by (device, stream), so that concurrent streams never share one.  A CUDA graph captured in this mode
// holds the capturing stream's buffers; a buffer that a larger call outgrows is therefore retired, not freed, and stays valid
// until mf_det_release() (which synchronises the devices and frees everything, so graphs captured in this mode must not be
// replayed after it).
// ---------------------------------------------------------------------------------------------
namespace {
struct DetSlot {
    int dev; cudaStream_t st;
    int64_t n_cap, p_cap;
    DetWs ws;
    std::vector<void*> retired;
    int64_t retired_bytes;
};
std::mutex g_det_mu;
std::vector<DetSlot> g_det_slots;

int64_t slot_bytes(const DetSlot& s) { return s.n_cap * MF_DET_ROW * 4 + s.p_cap * (4 + 8) + s.retired_bytes; }

void free_slot(DetSlot& s) {
    cudaFree(s.ws.rows); cudaFree(s.ws.expo); cudaFree(s.ws.acc);
    for (void* p : s.retired) cudaFree(p);
    s.ws = DetWs{}; s.n_cap = s.p_cap = 0; s.retired.clear(); s.retired_bytes = 0;
}
}  // namespace

int mf_det_workspace(int64_t n, int64_t P, cudaStream_t st, DetWs* ws) {
    int dev = 0;
    MF_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lk(g_det_mu);
    DetSlot* s = nullptr;
    for (auto& e : g_det_slots)
        if (e.dev == dev && e.st == st) { s = &e; break; }
    if (!s) { g_det_slots.push_back(DetSlot{dev, st, 0, 0, DetWs{}, {}, 0}); s = &g_det_slots.back(); }
    if (n > s->n_cap || P > s->p_cap) {
        cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
        MF_CUDA(cudaStreamIsCapturing(st, &cs));
        if (cs != cudaStreamCaptureStatusNone) {
            mf_set_error("deterministic mode: the workspace of this stream must grow to %lld points / %lld gradient floats during "
                         "stream capture; run the call once outside capture first", (long long)n, (long long)P);
            return MF_ERR_INVALID;
        }
        if (n > s->n_cap) {
            if (s->ws.rows) { s->retired.push_back(s->ws.rows); s->retired_bytes += s->n_cap * MF_DET_ROW * 4; }
            s->ws.rows = nullptr; s->n_cap = 0;
            MF_CUDA(cudaMalloc(&s->ws.rows, (size_t)n * MF_DET_ROW * sizeof(float)));
            s->n_cap = n;
        }
        if (P > s->p_cap) {
            if (s->ws.expo) {
                s->retired.push_back(s->ws.expo); s->retired.push_back(s->ws.acc); s->retired_bytes += s->p_cap * (4 + 8);
            }
            s->ws.expo = nullptr; s->ws.acc = nullptr; s->p_cap = 0;
            MF_CUDA(cudaMalloc(&s->ws.expo, (size_t)P * sizeof(uint32_t)));
            MF_CUDA(cudaMalloc(&s->ws.acc, (size_t)P * sizeof(unsigned long long)));
            MF_CUDA(cudaMemsetAsync(s->ws.expo, 0, (size_t)P * sizeof(uint32_t), st));
            MF_CUDA(cudaMemsetAsync(s->ws.acc, 0, (size_t)P * sizeof(unsigned long long), st));
            s->p_cap = P;
        }
    }
    *ws = s->ws;
    return MF_OK;
}

int mf_det_scatter(const FieldDev& f, const DetWs& ws, const float* x, int ldx, const float* dy, int ldy, const int* count, int64_t n,
                   float* grad, cudaStream_t st) {
    if (n <= 0) return MF_OK;
    const int h = 64 - __builtin_clzll((unsigned long long)n * 8ull);      // ceil(log2(8 n + 1))
    if (n >= ((int64_t)1 << 32) || h > MF_DET_MAX_H) {
        mf_set_error("deterministic mode: %lld points in one launch exceed the fixed-point headroom (at most 2^32 - 1)", (long long)n);
        return MF_ERR_INVALID;
    }
    const unsigned blocks = (unsigned)((n * f.n_levels + DET_NT - 1) / DET_NT);
    const int64_t P = 2 * ((int64_t)f.offset[f.n_levels - 1] + f.size[f.n_levels - 1]);
    MF_CUDA(mf_launch(det_pass1_kernel, blocks, DET_NT, 0, st, f, x, ldx, dy, ldy, count, n, ws.expo));
    MF_CUDA(mf_launch(det_pass2_kernel, blocks, DET_NT, 0, st, f, x, ldx, dy, ldy, count, n, h, ws.expo, ws.acc));
    MF_CUDA(mf_launch(det_finalize_kernel, (unsigned)(mf_sm_count_cached() * 8), DET_NT, 0, st, h, P, ws.expo, ws.acc, grad));
    return MF_OK;
}

MF_API int64_t mf_det_workspace_bytes(void) {
    std::lock_guard<std::mutex> lk(g_det_mu);
    int64_t b = 0;
    for (const auto& s : g_det_slots) b += slot_bytes(s);
    return b;
}

MF_API int mf_det_release(void) {
    std::lock_guard<std::mutex> lk(g_det_mu);
    int prev = 0;
    MF_CUDA(cudaGetDevice(&prev));
    for (auto& s : g_det_slots) {
        MF_CUDA(cudaSetDevice(s.dev));
        MF_CUDA(cudaDeviceSynchronize());
        free_slot(s);
    }
    g_det_slots.clear();
    MF_CUDA(cudaSetDevice(prev));
    return MF_OK;
}
