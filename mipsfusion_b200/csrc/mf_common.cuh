// Shared host/device helpers for the mipsfusion_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/mipsfusion_b200.h"

#define MF_API extern "C" __attribute__((visibility("default")))

void mf_set_error(const char* fmt, ...);

#define MF_CHECK_ARG(cond)                                                        \
    do {                                                                          \
        if (!(cond)) {                                                            \
            mf_set_error("%s: invalid argument: %s", __func__, #cond);            \
            return MF_ERR_INVALID;                                                \
        }                                                                         \
    } while (0)

#define MF_CUDA(expr)                                                             \
    do {                                                                          \
        cudaError_t _e = (expr);                                                  \
        if (_e != cudaSuccess) {                                                  \
            mf_set_error("%s: %s -> %s", __func__, #expr, cudaGetErrorString(_e)); \
            return MF_ERR_CUDA;                                                   \
        }                                                                         \
    } while (0)

#define MF_LAUNCH_CHECK() MF_CUDA(cudaGetLastError())

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (PDL).  mf_launch() issues a kernel with programmatic stream serialization (unless
// mf_set_pdl(0) or MF_NO_PDL=1 in the environment): its CTAs may be scheduled, and run their prologue, as soon as every CTA
// of the kernel before it in the stream has executed mf_pdl_trigger() or exited.  mf_pdl_wait() then blocks until that
// kernel has completed and its memory operations are visible.  Both instructions are no-ops in a kernel launched without
// the attribute, so the same kernels serve <<<>>> launches and stream capture unchanged.
//
// Hazard rule: mf_pdl_wait() orders a grid only against its IMMEDIATE predecessor.  A kernel launched through mf_launch()
// therefore touches no global memory (neither reads nor writes) before its mf_pdl_wait(), and every one of them executes it
// first thing.  Then each such kernel completes only after its predecessor has completed, completion is ordered
// transitively along the stream, and a buffer written two or more kernels back (the weight image from mlp_prepare, the
// forward's tile counter pair, the backward's active count, the gradients Adam zeroed) is complete when the wait returns.
// Moving work that reads such a buffer in front of the wait would be a race: the field kernels also run directly after
// mf_mlp_prepare (sync_to_module), and the predecessor's own trigger may precede its writes.  (Moving the TMEM / mbarrier
// set-up of the field kernels in front of the wait was tried: it added spills to the forward kernel.)
// mf_pdl_trigger() only lets the next grid's CTAs be scheduled; the small kernels issue it right after their wait (their
// grids fit on the GPU in one wave), the persistent 1-CTA/SM field kernels after the CTA's last tile.
// Event records between two kernels (mapper.timing, mf_debug_kernel_timer) end the overlap; results are unaffected.
// ---------------------------------------------------------------------------------------------
bool mf_pdl_enabled();

template <typename... KArgs, typename... Args>
static inline cudaError_t mf_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cfg.attrs = attr; cfg.numAttrs = mf_pdl_enabled() ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

__device__ __forceinline__ void mf_pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void mf_pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

int mf_sm_count_cached();
constexpr int MF_KTIMER_SLOTS = 4;
void mf_ktimer_begin(int slot, cudaStream_t st);   // no-ops unless mf_debug_kernel_timer(1)
void mf_ktimer_end(int slot, cudaStream_t st);

// ---------------------------------------------------------------------------------------------
// Tile geometry of the fused field kernels: one CTA works on TP points at a time; activations
// live in shared memory feature-major, act[k][m] with a padded row of LDA floats so that rows
// k, k+1, ... fall 4 banks apart (conflict-free float4 access for 16 consecutive rows).
// ---------------------------------------------------------------------------------------------
constexpr int TP = 64;            // points per tile
constexpr int LDA = TP + 4;       // padded row length (floats)
constexpr int NT = 256;           // threads per CTA

// Decoder dimensions (reference model/decoder.py:6-50 as instantiated by model/scene_rep.py:45).
constexpr int D_GRID = 32;        // hash-grid features
constexpr int D_FREQ = 48;        // frequency features
constexpr int D_E = 51;           // [xyz(3), freq(48)]
constexpr int D_EP = 52;          // padded
constexpr int D_H = 128;          // hidden
constexpr int D_SDF_EMB = 64;
constexpr int D_RGB_IN = 115;     // [rgb_emb(64), e(51)]
constexpr int D_SDF_IN = 96;      // [sdf_emb(64), grid(32)]
constexpr int N_CLASS = 5;

// Offsets into the flat state_dict-ordered parameter blob (`mlp`, MF_MLP_PARAMS floats).
constexpr int OFF_W1 = 0;                         // (128,51)
constexpr int OFF_B1 = OFF_W1 + 128 * 51;
constexpr int OFF_W2 = OFF_B1 + 128;              // (128,128)
constexpr int OFF_B2 = OFF_W2 + 128 * 128;
constexpr int OFF_WR = OFF_B2 + 128;              // (3,115)
constexpr int OFF_BR = OFF_WR + 3 * 115;
constexpr int OFF_WS1 = OFF_BR + 3;               // (128,96)
constexpr int OFF_BS1 = OFF_WS1 + 128 * 96;
constexpr int OFF_WS2 = OFF_BS1 + 128;            // (5,128)
constexpr int OFF_BS2 = OFF_WS2 + 5 * 128;
static_assert(OFF_BS2 + 5 == MF_MLP_PARAMS, "decoder parameter count");

// Kernel-layout weights (`mlp_prep`): the original blob followed by permuted copies.
//   forward  copy  F_l[k][tx][i] = W_l[n = tx + 16 i][k]      (k-major, 128 outputs)
//   backward copy  B_l[n][tx][i] = W_l[n][k = tx + 16 i]      (n-major, KI = ceil(K/16) per tx, zero padded)
constexpr int PREP_RAW = 0;
constexpr int PREP_F1 = 36608;                    // 52 x 128   (row 51 zero)
constexpr int PREP_F2 = PREP_F1 + 52 * 128;       // 128 x 128
constexpr int PREP_F3 = PREP_F2 + 128 * 128;      // 96 x 128
constexpr int PREP_B1 = PREP_F3 + 96 * 128;       // 128 x 64   (KI = 4)
constexpr int PREP_B2 = PREP_B1 + 128 * 64;       // 128 x 128  (KI = 8)
constexpr int PREP_B3 = PREP_B2 + 128 * 128;      // 128 x 96   (KI = 6)
constexpr int PREP_SIMT_SIZE = PREP_B3 + 128 * 96;
constexpr int PREP_TC = PREP_SIMT_SIZE;           // tensor-core weight image (field_tc.cuh), 169,552 bytes
constexpr int PREP_SIZE = PREP_TC + 42388;
static_assert(PREP_F1 >= MF_MLP_PARAMS && PREP_F1 % 4 == 0 && PREP_TC % 4 == 0, "alignment");

// Device-side copy of mf_grid_meta + normalisation, passed by value as a kernel parameter.
struct FieldDev {
    const float* grid;
    const float* prep;
    const uint8_t* tc_img;        // prep + PREP_TC: bf16 hi/lo weight image of the tcgen05 decoder
    uint32_t* feat;               // optional encoded-feature cache written by the tc forward, read by the tc backward
    double na[3], nb[3], nf;
    int impl;                     // resolved decoder implementation: 0 tcgen05, 1 fp32 CUDA cores
    int n_levels;
    float scale[MF_MAX_LEVELS];
    uint32_t res[MF_MAX_LEVELS], size[MF_MAX_LEVELS], offset[MF_MAX_LEVELS], hashed[MF_MAX_LEVELS];
};

// Backward kernels only visit the points whose upstream gradient row is non-zero ("active" points; the others add
// exactly zero to every gradient).  idx (ascending point indices) and count live in the caller's workspace and are
// written by compact_active_points(); idx == nullptr is the identity map over [0, N).
struct ActiveMap {
    const int* idx; const int* count;
    __device__ __forceinline__ int64_t n(int64_t N) const { return count ? (int64_t)*count : N; }
    __device__ __forceinline__ int64_t operator()(int64_t slot) const { return idx ? (int64_t)idx[slot] : slot; }
};

// ---------------------------------------------------------------------------------------------
// Deterministic mode (mf_set_deterministic, det_kernels.cu).  The backward kernels' deterministic instantiations (point source
// DetRows<Src>, field_core.cuh) do not scatter into the table: they write one row of MF_DET_ROW floats per active slot -- the
// normalised position at [0, 3), the 32 grid-feature gradients at [MF_DET_DY, MF_DET_DY + 32) -- and mf_det_scatter forms
// grad += sum of the contributions by fixed-point accumulation, whose result depends only on the multiset of contributions.
// ---------------------------------------------------------------------------------------------
constexpr int MF_DET_ROW = 36;
constexpr int MF_DET_DY = 4;
constexpr int MF_DET_MAX_H = 35;      // headroom bits: 8 N + 1 <= 2^35 (N < 2^32 points per launch)
bool mf_deterministic();
struct DetWs {
    float* rows;                      // [n][MF_DET_ROW]
    uint32_t* expo;                   // [P] per gradient float: max exponent of its contributions | non-finite flags (zero between calls)
    unsigned long long* acc;          // [P] fixed-point sums (zero between calls)
};
// The library-owned workspace of (current device, st) with room for n rows and P gradient floats; grows outside stream
// capture only (an error under capture).  Outgrown buffers are retired, not freed, until mf_det_release (captured graphs).
int mf_det_workspace(int64_t n, int64_t P, cudaStream_t st, DetWs* ws);
// grad[e] += sum of __fmul_rn(w, dy) over the (point, level, corner) contributions to e of the n points (x[i * ldx + d],
// dy[i * ldy + 2 l + k]); count (device, may be NULL) limits the points to its value.  Three kernels through mf_launch.
int mf_det_scatter(const FieldDev& f, const DetWs& ws, const float* x, int ldx, const float* dy, int ldy, const int* count, int64_t n,
                   float* grad, cudaStream_t st);
// dx (N, 3) of the stand-alone hash-grid encoding (16 levels) without the table scatter
int mf_det_hashgrid_dx(const FieldDev& f, const float* x, const float* dy, float* dx, int64_t N, cudaStream_t st);

int mf_field_to_dev(const mf_field* f, FieldDev* d);   // validates (16 levels, 2 features)
int mf_decoder_impl();                                 // 0: tcgen05 tensor cores (default), 1: fp32 CUDA cores
int mf_bwd_impl();                                     // tensor-core backward: 0 role-split kernel (default), 1 single-role kernel
int* mf_tc_error_flag();
// {next tile, CTAs done} pair for one launch of a kernel with dynamic tile scheduling (zero on entry, re-armed by the last CTA of
// the launch); drawn round-robin from a per-device ring, so launches in flight on different streams do not share a pair.
// mf_set_dynamic_tiles(0) -> NULL (static striding, A/B).
int* mf_tile_counter();
int mf_sm_reserve();
constexpr int MF_PROF_SLOTS = 1024;
long long* mf_tc_profile_buffer();
__device__ __forceinline__ long long mf_globaltimer() { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; }                     // device buffer of 64 clock stamps, or nullptr when profiling is off                               // device int, set by a kernel whose MMA wait timed out

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ int warp_min_i(int v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = min(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }
