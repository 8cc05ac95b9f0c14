// Multi-resolution hash grid: index arithmetic, gather, scatter and input gradient.
// Restates the published algorithm of tinycudann 1.7 (encodings/grid.h) that the reference
// selects at model/encodings.py:14-25 -- see oracle/hashgrid.py for the normative definition.
#pragma once
#include "mf_common.cuh"

constexpr uint32_t MF_PRIME1 = 2654435761u;
constexpr uint32_t MF_PRIME2 = 805459861u;

struct LevelInfo {
    float scale;
    uint32_t res, size, offset, hashed;
};

__device__ __forceinline__ LevelInfo level_info(const FieldDev& f, int l) {
    LevelInfo li;
    li.scale = f.scale[l]; li.res = f.res[l]; li.size = f.size[l]; li.offset = f.offset[l]; li.hashed = f.hashed[l];
    return li;
}

// grid_index<3, CoherentPrime>: all arithmetic is uint32 with wrap-around.
__device__ __forceinline__ uint32_t grid_index(uint32_t px, uint32_t py, uint32_t pz, const LevelInfo& li) {
    uint32_t idx;
    if (li.hashed) {
        idx = px ^ (py * MF_PRIME1) ^ (pz * MF_PRIME2);
    } else {
        idx = px + py * li.res + pz * (li.res * li.res);
    }
    if (idx >= li.size) idx %= li.size;
    return idx;
}

// pos_fract(): pos = fmaf(scale, x, 0.5); cell = (uint32)(int)floor(pos); frac = pos - floor(pos)
__device__ __forceinline__ void pos_fract(float x, float scale, uint32_t& cell, float& frac) {
    float pos = fmaf(scale, x, 0.5f);
    float fl = floorf(pos);
    cell = (uint32_t)(int)fl;
    frac = pos - fl;
}

// The 8 corner indices and trilinear weights of one level.  Same arithmetic as grid_index / the tcnn corner loop
// (uint32 wrap-around; weight = ((1 * w_x) * w_y) * w_z), with the per-dimension terms computed once.  Hashed
// levels always have a power-of-two size (2^log2_hashmap_size), so their modulo is a mask.
__device__ __forceinline__ void grid_corners(const float x[3], const LevelInfo& li, uint32_t (&idx)[8], float (&w)[8]) {
    uint32_t g[3]; float f[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) pos_fract(x[d], li.scale, g[d], f[d]);
    uint32_t tx[2], ty[2], tz[2];
    tx[0] = g[0]; tx[1] = g[0] + 1u;
    if (li.hashed) {
        ty[0] = g[1] * MF_PRIME1; ty[1] = (g[1] + 1u) * MF_PRIME1;
        tz[0] = g[2] * MF_PRIME2; tz[1] = (g[2] + 1u) * MF_PRIME2;
        const uint32_t mask = li.size - 1u;
#pragma unroll
        for (int c = 0; c < 8; ++c) idx[c] = (tx[c & 1] ^ ty[(c >> 1) & 1] ^ tz[(c >> 2) & 1]) & mask;
    } else {
        const uint32_t r2 = li.res * li.res;
        ty[0] = g[1] * li.res; ty[1] = (g[1] + 1u) * li.res;
        tz[0] = g[2] * r2; tz[1] = (g[2] + 1u) * r2;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
            uint32_t i = tx[c & 1] + ty[(c >> 1) & 1] + tz[(c >> 2) & 1];
            if (i >= li.size) i %= li.size;
            idx[c] = i;
        }
    }
    const float wx[2] = {__fsub_rn(1.0f, f[0]), f[0]}, wy[2] = {__fsub_rn(1.0f, f[1]), f[1]}, wz[2] = {__fsub_rn(1.0f, f[2]), f[2]};
#pragma unroll
    for (int c = 0; c < 8; ++c) w[c] = __fmul_rn(__fmul_rn(wx[c & 1], wy[(c >> 1) & 1]), wz[(c >> 2) & 1]);
}

#ifndef MF_PAIR_GATHER
#define MF_PAIR_GATHER 0
#endif
// Forward gather of one level: 8 corners, 2 features.  idx_out (8) optional.
__device__ __forceinline__ float2 grid_level_fwd(const float x[3], const float2* __restrict__ grid2,
                                                 const LevelInfo& li, uint32_t* idx_out) {
    uint32_t idx[8]; float w[8];
    grid_corners(x, li, idx, w);
    float2 v[8];
#if MF_PAIR_GATHER
    // x-neighbours (idx[2k], idx[2k+1]) that are table neighbours on a 16-byte boundary (even x on a dense level without wrap,
    // even x on a hashed level: (x + 1) ^ h = (x ^ h) ^ 1) come in with ONE 16-byte gather: fewer load wavefronts per point
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint32_t i0 = idx[2 * k], i1 = idx[2 * k + 1];
        if (((i0 & 1u) == 0u) && (i1 == i0 + 1u)) {
            const float4 q = __ldg(reinterpret_cast<const float4*>(&grid2[li.offset + i0]));
            v[2 * k] = make_float2(q.x, q.y); v[2 * k + 1] = make_float2(q.z, q.w);
        } else {
            v[2 * k] = __ldg(&grid2[li.offset + i0]); v[2 * k + 1] = __ldg(&grid2[li.offset + i1]);
        }
    }
#else
#pragma unroll
    for (int c = 0; c < 8; ++c) v[c] = __ldg(&grid2[li.offset + idx[c]]);     // 8 independent gathers in flight
#endif
    float2 acc = make_float2(0.f, 0.f);
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        acc.x = fmaf(w[c], v[c].x, acc.x);
        acc.y = fmaf(w[c], v[c].y, acc.y);
        if (idx_out) idx_out[c] = idx[c];
    }
    return acc;
}

__device__ __forceinline__ void red_add_f2(float* addr, float a, float b) {
    asm volatile("red.global.add.v2.f32 [%0], {%1, %2};" ::"l"(addr), "f"(a), "f"(b) : "memory");
}

__device__ __forceinline__ void red_add_f4(float* addr, float a, float b, float c, float d) {
    asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(addr), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

// Backward of one level: scatter w * dy into grad (kernel_grid_backward) and, if WANT_DX,
// return dL/dx contribution (kernel_grid_backward_input; needs the forward features).
// SCATTER = false: input gradient only (pose refinement: no parameter gradients wanted).
template <bool WANT_DX, bool SCATTER = true>
__device__ __forceinline__ void grid_level_bwd(const float x[3], float2 dy, const float2* __restrict__ grid2,
                                               float* __restrict__ grad, const LevelInfo& li, float dx[3]) {
    uint32_t idx[8]; float w8[8];
    grid_corners(x, li, idx, w8);
    if (SCATTER && (dy.x != 0.f || dy.y != 0.f)) {
        // the two corners of an x-pair are neighbours in the table whenever their indices differ only in bit 0 (cell x even
        // on a hashed level, even linear index on a dense one; level offsets are multiples of 8): one 16-byte reduction
        // instead of two 8-byte ones -- the scatter is bound by reduction lanes per SM
#pragma unroll
        for (int c = 0; c < 8; c += 2) {
            const uint32_t i0 = idx[c], i1 = idx[c + 1];
            if ((i0 ^ i1) == 1u) {
                const bool sw = (i0 & 1u) != 0u;                       // i1 is the even (lower) entry
                const float wa = sw ? w8[c + 1] : w8[c], wb = sw ? w8[c] : w8[c + 1];
                red_add_f4(grad + 2 * (size_t)(li.offset + (i0 & ~1u)), wa * dy.x, wa * dy.y, wb * dy.x, wb * dy.y);
            } else {
                red_add_f2(grad + 2 * (size_t)(li.offset + i0), w8[c] * dy.x, w8[c] * dy.y);
                red_add_f2(grad + 2 * (size_t)(li.offset + i1), w8[c + 1] * dy.x, w8[c + 1] * dy.y);
            }
        }
    }
    if (WANT_DX) {
        float f[3];
#pragma unroll
        for (int d = 0; d < 3; ++d) { uint32_t gd; pos_fract(x[d], li.scale, gd, f[d]); }
        float2 v[8];
#pragma unroll
        for (int c = 0; c < 8; ++c) v[c] = __ldg(&grid2[li.offset + idx[c]]);
#pragma unroll
        for (int d = 0; d < 3; ++d) {
            // d/dx_d of the trilinear blend: scale * sum over the 4 corner pairs along d
            const int d1 = (d + 1) % 3, d2 = (d + 2) % 3;
            float s = 0.f;
#pragma unroll
            for (int a = 0; a < 2; ++a)
#pragma unroll
                for (int b = 0; b < 2; ++b) {
                    float w = (a ? f[d1] : 1.0f - f[d1]) * (b ? f[d2] : 1.0f - f[d2]);
                    int c0 = (a << d1) | (b << d2);
                    int c1 = c0 | (1 << d);
                    s += w * ((v[c1].x - v[c0].x) * dy.x + (v[c1].y - v[c0].y) * dy.y);
                }
            dx[d] += li.scale * s;
        }
    }
}

// Backward of the stand-alone encoding (mf_hashgrid_bwd): thread per (point, level).
template <bool WANT_DX, bool SCATTER>
__device__ __forceinline__ void hashgrid_bwd_body(const FieldDev& f, const float* __restrict__ x, const float* __restrict__ dy,
                                                  float* __restrict__ grad, float* __restrict__ dx_out, int64_t N) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int L = f.n_levels;                       // 16 levels -> the 16 lanes of a half warp share a point
    const bool active = t < N * L;
    const int64_t i = active ? t / L : 0; const int l = (int)(t % L);
    float dx[3] = {0.f, 0.f, 0.f};
    if (active) {
        const float xv[3] = {x[i * 3], x[i * 3 + 1], x[i * 3 + 2]};
        const float2 g = reinterpret_cast<const float2*>(dy)[t];
        grid_level_bwd<WANT_DX, SCATTER>(xv, g, reinterpret_cast<const float2*>(f.grid), grad, level_info(f, l), dx);
    }
    if (WANT_DX) {
#pragma unroll
        for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) dx[d] += __shfl_xor_sync(0xffffffffu, dx[d], o);
        if (active && l == 0) { dx_out[i * 3] = dx[0]; dx_out[i * 3 + 1] = dx[1]; dx_out[i * 3 + 2] = dx[2]; }
    }
}

// Warp-aggregated scatter of one level (all 32 lanes of the warp call it together; lane = point, consecutive lanes = consecutive
// active points = mostly consecutive samples of one ray).  Consecutive samples share their cell on the coarse levels -- the samples
// a loss term sees sit within the truncation distance of the surface, a few centimetres apart -- so lanes are grouped into runs of
// equal cell (compare with the previous lane, one ballot), the eight corner contributions are summed along each run with a
// segmented shuffle scan (as many doubling steps as the longest run needs; none when every run has length one), and only the
// last lane of a run issues the reductions: the SM's reduction rate is per lane (1.29 cycles), a shuffle step is not.
// Same values as grid_level_bwd up to the order of the float additions (the atomics already leave that order open).
__device__ __forceinline__ void grid_level_scatter_agg(const float x[3], float2 dy, float* __restrict__ grad, const LevelInfo& li, int lane) {
    constexpr uint32_t FULL = 0xffffffffu;
    uint32_t g[3]; float fr[3];
#pragma unroll
    for (int d = 0; d < 3; ++d) pos_fract(x[d], li.scale, g[d], fr[d]);
    const bool same = (__shfl_up_sync(FULL, g[0], 1) == g[0]) & (__shfl_up_sync(FULL, g[1], 1) == g[1]) & (__shfl_up_sync(FULL, g[2], 1) == g[2]);
    const uint32_t heads = __ballot_sync(FULL, lane == 0 || !same);
    const int off = lane - (31 - __clz((int)(heads & (FULL >> (31 - lane)))));       // distance to the head of this lane's run
    const bool tail = lane == 31 || ((heads >> (lane + 1)) & 1u);
    uint32_t idx[8]; float w8[8];
    grid_corners(x, li, idx, w8);
    float vx[8], vy[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) { vx[c] = w8[c] * dy.x; vy[c] = w8[c] * dy.y; }
    if (heads != FULL) {                                   // (warp-uniform)
#pragma unroll 1
        for (int d = 1; d < 32; d <<= 1) {
            if (!__any_sync(FULL, off >= d)) break;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
                const float ax = __shfl_up_sync(FULL, vx[c], d), ay = __shfl_up_sync(FULL, vy[c], d);
                if (off >= d) { vx[c] += ax; vy[c] += ay; }
            }
        }
    }
    if (tail) {
#pragma unroll
        for (int c = 0; c < 8; c += 2) {                   // x-pairs that are table neighbours leave as one 16-byte reduction (grid_level_bwd)
            if (vx[c] == 0.f && vy[c] == 0.f && vx[c + 1] == 0.f && vy[c + 1] == 0.f) continue;
            const uint32_t i0 = idx[c], i1 = idx[c + 1];
            if ((i0 ^ i1) == 1u) {
                const bool sw = (i0 & 1u) != 0u;
                red_add_f4(grad + 2 * (size_t)(li.offset + (i0 & ~1u)), sw ? vx[c + 1] : vx[c], sw ? vy[c + 1] : vy[c], sw ? vx[c] : vx[c + 1],
                           sw ? vy[c] : vy[c + 1]);
            } else {
                red_add_f2(grad + 2 * (size_t)(li.offset + i0), vx[c], vy[c]);
                red_add_f2(grad + 2 * (size_t)(li.offset + i1), vx[c + 1], vy[c + 1]);
            }
        }
    }
}

// Coordinate normalisation of JointEncoding.run_network (model/scene_rep.py:138-142) followed by
// "/ norm_factor" (:119): fp64 arithmetic, one rounding to fp32 (the bound tensors are float64).
__device__ __forceinline__ void normalize_point(const FieldDev& f, const float p[3], float x[3]) {
#pragma unroll
    for (int d = 0; d < 3; ++d) x[d] = (float)((((double)p[d] - f.na[d]) / f.nb[d]) / f.nf);
}
__device__ __forceinline__ void prenormalized_point(const FieldDev& f, const float p[3], float x[3]) {
#pragma unroll
    for (int d = 0; d < 3; ++d) x[d] = (f.nf == 1.0) ? p[d] : __fdiv_rn(p[d], (float)f.nf);   // fp32 tensor / python scalar
}

// Frequency encoding argument: fl(fl(x * 2^k) * PI) (+ fl(PI/2)); oracle/frequency.py.
__device__ __forceinline__ float freq_arg(float x, int k, int s) {
    float a = __fmul_rn(ldexpf(x, k), 3.14159274101257324f);
    return s ? __fadd_rn(a, 1.57079637050628662f) : a;
}

// sin(arg) for the tensor-core kernels: explicit three-term Cody-Waite reduction to [-pi, pi] followed by the
// MUFU approximation (abs error ~5e-7 for |arg| <= 128 pi + pi/2, the range of the frequency encoding).  The
// argument is the same fp32 number the oracle feeds to torch.sin; only the evaluation is cheaper than sinf().
__device__ __forceinline__ float sin_reduced(float arg) {
    const float k = rintf(arg * 0.15915494309189535f);
    float r = fmaf(k, -6.28318548202514648f, arg);          // 2 pi = hi + mid + lo
    r = fmaf(k, 1.74845553146951715e-7f, r);
    r = fmaf(k, 7.1054274e-15f, r);
    return __sinf(r);
}
__device__ __forceinline__ float cos_reduced(float arg) {
    const float k = rintf(arg * 0.15915494309189535f);
    float r = fmaf(k, -6.28318548202514648f, arg);
    r = fmaf(k, 1.74845553146951715e-7f, r);
    r = fmaf(k, 7.1054274e-15f, r);
    return __cosf(r);
}
