// Fused per-tile field evaluation: normalise -> hash-grid + frequency encode -> MLP_reg decoder,
// forward and backward, for one tile of TP points held feature-major in shared memory.
//
// This is the fp32 CUDA-core (SIMT) implementation of the decoder GEMMs.  It is exact fp32
// (FMA accumulation) and is the numerical reference for the tensor-core path.
//
// Reference semantics: model/scene_rep.py:118-146 (query), model/decoder.py:53-75 (decoder),
// tinycudann 1.7 grid/frequency encodings (oracle/hashgrid.py, oracle/frequency.py).
#pragma once
#include "grid_encode.cuh"

// Shared-memory rows (each LDA floats).
constexpr int ROW_E = 0;                 // 52 rows: x(3), freq(48), zero pad
constexpr int ROW_G = ROW_E + D_EP;      // 32 rows: grid features
constexpr int ROW_H1 = ROW_G + D_GRID;   // 128 rows
constexpr int ROW_H2 = ROW_H1 + D_H;     // 128 rows
constexpr int ROW_SM = ROW_H2 + D_H;     // 32 rows of partial sums + 10 rows of outputs + 2 spare
constexpr int ROW_OUT = ROW_SM + 32;
constexpr int ROWS_FWD = ROW_SM + 44;
constexpr int ROW_H3 = ROWS_FWD;         // backward only: 128 rows
constexpr int ROW_DZ = ROW_H3 + D_H;     // backward only: 8 rows (dlogits 5, drgb 3)
constexpr int ROWS_BWD = ROW_DZ + 8;
constexpr size_t SMEM_FWD = (size_t)ROWS_FWD * LDA * sizeof(float);
constexpr size_t SMEM_BWD = (size_t)ROWS_BWD * LDA * sizeof(float);

// ------------------------------------------------------------------------------------------
// Point sources: produce the (already normalised) encoder input x for global point index i.
// ------------------------------------------------------------------------------------------
struct SrcPoints {                       // explicit points in the submap frame
    const float* pts; int normalize;
    __device__ __forceinline__ void point(int64_t i, const FieldDev& f, float x[3]) const {
        float p[3] = {pts[i * 3 + 0], pts[i * 3 + 1], pts[i * 3 + 2]};
        if (normalize) normalize_point(f, p, x); else prenormalized_point(f, p, x);
    }
    __device__ __forceinline__ void dx_to_dp(const FieldDev& f, const float dx[3], float dp[3]) const {
#pragma unroll
        for (int d = 0; d < 3; ++d) dp[d] = normalize ? (float)((double)dx[d] / (f.nb[d] * f.nf)) : (float)((double)dx[d] / f.nf);
    }
};

struct SrcRays {                         // pts = rays_o + rays_d * z   (model/scene_rep.py:179), fp32 mul then add
    const float* o; const float* d; const float* z; int S;
    __device__ __forceinline__ void point(int64_t i, const FieldDev& f, float x[3]) const {
        int64_t r = i / S;
        float zz = z[i];
        float p[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) p[k] = __fadd_rn(o[r * 3 + k], __fmul_rn(d[r * 3 + k], zz));
        normalize_point(f, p, x);
    }
    __device__ __forceinline__ void dx_to_dp(const FieldDev& f, const float dx[3], float dp[3]) const {
#pragma unroll
        for (int d_ = 0; d_ < 3; ++d_) dp[d_] = (float)((double)dx[d_] / (f.nb[d_] * f.nf));
    }
};

// Point source of the deterministic backward instantiations (mf_common.cuh): the same points, but the kernel writes the
// grid-gradient rows to grad_grid (the row buffer) instead of scattering.  A distinct type rather than a kernel parameter, so
// that the default instantiations keep their code and registers.
template <class S> struct DetRows : S {};
template <class S> struct is_det_rows { static constexpr bool value = false; };
template <class S> struct is_det_rows<DetRows<S>> { static constexpr bool value = true; };

__device__ __forceinline__ void det_store_x(float* rows, int64_t slot, const float x[3]) {
    *reinterpret_cast<float4*>(rows + slot * MF_DET_ROW) = make_float4(x[0], x[1], x[2], 0.f);
}
// the whole row: x and the 32 gradient words (role-split backward, field_tc_bwd2.cuh)
__device__ __forceinline__ void det_store_row(float* rows, int64_t slot, const float x[3], const uint32_t (&r)[32]) {
    float4* row = reinterpret_cast<float4*>(rows + slot * MF_DET_ROW);
    row[0] = make_float4(x[0], x[1], x[2], 0.f);
#pragma unroll
    for (int j = 0; j < 8; ++j)
        row[1 + j] = make_float4(__uint_as_float(r[4 * j]), __uint_as_float(r[4 * j + 1]), __uint_as_float(r[4 * j + 2]), __uint_as_float(r[4 * j + 3]));
}
// the gradients of levels 4 q .. 4 q + 3
__device__ __forceinline__ void det_store_dy8(float* rows, int64_t slot, int q, const float dy[8]) {
    float4* r = reinterpret_cast<float4*>(rows + slot * MF_DET_ROW + MF_DET_DY + 8 * q);
    r[0] = make_float4(dy[0], dy[1], dy[2], dy[3]);
    r[1] = make_float4(dy[4], dy[5], dy[6], dy[7]);
}

// ------------------------------------------------------------------------------------------
// Encode one tile: thread (m = tid & 63, q = tid >> 6) handles 4 grid levels and 12 frequency
// outputs of point m.
// ------------------------------------------------------------------------------------------
template <class Src>
__device__ __forceinline__ void encode_tile(const FieldDev& f, const Src& src, int64_t tile, int64_t N, float* sm,
                                            const ActiveMap am = ActiveMap{nullptr, nullptr}) {
    const int tid = threadIdx.x, m = tid & (TP - 1), q = tid >> 6;
    const int64_t slot = tile * TP + m;
    const bool valid = slot < N;
    const int64_t i = valid ? am(slot) : 0;
    float x[3] = {0.f, 0.f, 0.f};
    if (valid) src.point(i, f, x);
    float* E = sm + ROW_E * LDA;
    float* G = sm + ROW_G * LDA;
    if (q == 0) {
        E[0 * LDA + m] = x[0]; E[1 * LDA + m] = x[1]; E[2 * LDA + m] = x[2];
        E[51 * LDA + m] = 0.f;
    }
#pragma unroll
    for (int jj = 0; jj < 12; ++jj) {
        const int j = q * 12 + jj, d = j >> 4, k = (j & 15) >> 1, s = j & 1;
        E[(3 + j) * LDA + m] = sinf(freq_arg(x[d], k, s));
    }
    const float2* grid2 = reinterpret_cast<const float2*>(f.grid);
#pragma unroll
    for (int ll = 0; ll < 4; ++ll) {
        const int l = q * 4 + ll;
        float2 v = make_float2(0.f, 0.f);
        if (valid) v = grid_level_fwd(x, grid2, level_info(f, l), nullptr);
        G[(2 * l) * LDA + m] = v.x;
        G[(2 * l + 1) * LDA + m] = v.y;
    }
}

// Features supplied by the caller (stand-alone MLP_reg.forward): embed (N,32), embed_pos (N,48), pts (N,3).
__device__ __forceinline__ void load_features_tile(const float* embed, const float* embed_pos, const float* pts,
                                                   int64_t tile, int64_t N, float* sm) {
    float* E = sm + ROW_E * LDA;
    float* G = sm + ROW_G * LDA;
    const int64_t base = tile * TP;
    const int nv = (int)min((int64_t)TP, N - base);
    for (int idx = threadIdx.x; idx < TP * D_GRID; idx += NT) {
        int m = idx / D_GRID, k = idx % D_GRID;
        G[k * LDA + m] = m < nv ? embed[(base + m) * D_GRID + k] : 0.f;
    }
    for (int idx = threadIdx.x; idx < TP * D_FREQ; idx += NT) {
        int m = idx / D_FREQ, k = idx % D_FREQ;
        E[(3 + k) * LDA + m] = m < nv ? embed_pos[(base + m) * D_FREQ + k] : 0.f;
    }
    for (int idx = threadIdx.x; idx < TP * 4; idx += NT) {
        int m = idx >> 2, k = idx & 3;
        if (k < 3) E[k * LDA + m] = m < nv ? pts[(base + m) * 3 + k] : 0.f;
        else E[51 * LDA + m] = 0.f;
    }
}

// ------------------------------------------------------------------------------------------
// SIMT GEMM cores.  Thread (tx = tid & 15, ty = tid >> 4) owns points m0..m0+3 (m0 = 4 ty) and
// outputs n = tx + 16 i.
// ------------------------------------------------------------------------------------------
// acc[mi][i] += sum_k A[k][m0+mi] * W[n = tx+16i][k], W given k-major permuted: Wf[(k*16+tx)*8 + i]
template <int K>
__device__ __forceinline__ void gemm_fwd_acc(float (&acc)[4][8], const float* __restrict__ A,
                                             const float* __restrict__ Wf, int tx, int m0) {
#pragma unroll 4
    for (int k = 0; k < K; ++k) {
        const float4 a = *reinterpret_cast<const float4*>(A + k * LDA + m0);
        const float4* wp = reinterpret_cast<const float4*>(Wf + (k * 16 + tx) * 8);
        const float4 w0 = __ldg(wp), w1 = __ldg(wp + 1);
        const float av[4] = {a.x, a.y, a.z, a.w};
        const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[mi][i] = fmaf(av[mi], wv[i], acc[mi][i]);
    }
}

// dgrad: acc[mi][i] += sum_n dZ[n][m0+mi] * W[n][k = tx+16i], W given n-major permuted: Wb[(n*16+tx)*KI + i]
template <int KI>
__device__ __forceinline__ void gemm_dgrad_acc(float (&acc)[4][KI], const float* __restrict__ dZ,
                                               const float* __restrict__ Wb, int tx, int m0) {
#pragma unroll 4
    for (int n = 0; n < D_H; ++n) {
        const float4 a = *reinterpret_cast<const float4*>(dZ + n * LDA + m0);
        const float2* wp = reinterpret_cast<const float2*>(Wb + (n * 16 + tx) * KI);
        float wv[KI];
#pragma unroll
        for (int i = 0; i < KI / 2; ++i) { float2 w = __ldg(wp + i); wv[2 * i] = w.x; wv[2 * i + 1] = w.y; }
        const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int i = 0; i < KI; ++i) acc[mi][i] = fmaf(av[mi], wv[i], acc[mi][i]);
    }
}

template <bool RELU>
__device__ __forceinline__ void store_acc(const float (&acc)[4][8], float* __restrict__ Z, int tx, int m0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        float4 v = make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]);
        if (RELU) { v.x = fmaxf(v.x, 0.f); v.y = fmaxf(v.y, 0.f); v.z = fmaxf(v.z, 0.f); v.w = fmaxf(v.w, 0.f); }
        *reinterpret_cast<float4*>(Z + (tx + 16 * i) * LDA + m0) = v;
    }
}

__device__ __forceinline__ void init_bias(float (&acc)[4][8], const float* __restrict__ b, int tx) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const float bv = __ldg(b + tx + 16 * i);
#pragma unroll
        for (int mi = 0; mi < 4; ++mi) acc[mi][i] = bv;
    }
}

// wgrad: gW[n][k] += sum_m dZ[n][m] * A[k][m] for n = ty + 16 j, k = tx + 16 i (< Kreal);
// rowp(k) returns the shared-memory row holding input feature k.  gW is this CTA's private
// partial (global, (out,in) layout), so plain read-modify-write is race-free.
template <int KI, class RowFn>
__device__ __forceinline__ void wgrad_tile(const float* __restrict__ dZ, RowFn rowp, int Kreal,
                                           float* __restrict__ gW, int tid) {
    const int tx = tid & 15, ty = tid >> 4;
    float acc[8][KI];
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int i = 0; i < KI; ++i) acc[j][i] = 0.f;
    const float* arow[KI];
#pragma unroll
    for (int i = 0; i < KI; ++i) arow[i] = (tx + 16 * i < Kreal) ? rowp(tx + 16 * i) : nullptr;
#pragma unroll 2
    for (int m = 0; m < TP; m += 4) {
        float4 a[KI];
#pragma unroll
        for (int i = 0; i < KI; ++i)
            a[i] = arow[i] ? *reinterpret_cast<const float4*>(arow[i] + m) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float4 z = *reinterpret_cast<const float4*>(dZ + (ty + 16 * j) * LDA + m);
#pragma unroll
            for (int i = 0; i < KI; ++i) {
                acc[j][i] = fmaf(z.x, a[i].x, acc[j][i]);
                acc[j][i] = fmaf(z.y, a[i].y, acc[j][i]);
                acc[j][i] = fmaf(z.z, a[i].z, acc[j][i]);
                acc[j][i] = fmaf(z.w, a[i].w, acc[j][i]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int i = 0; i < KI; ++i) {
            const int k = tx + 16 * i;
            if (k < Kreal) gW[(ty + 16 * j) * Kreal + k] += acc[j][i];
        }
}

// gB[n] += sum_m dZ[n][m], n < 128 (threads 0..127)
__device__ __forceinline__ void bias_grad_tile(const float* __restrict__ dZ, float* __restrict__ gB, int tid) {
    if (tid < D_H) {
        float s = 0.f;
#pragma unroll 4
        for (int m = 0; m < TP; m += 4) {
            const float4 z = *reinterpret_cast<const float4*>(dZ + tid * LDA + m);
            s += (z.x + z.y) + (z.z + z.w);
        }
        gB[tid] += s;
    }
}

// ------------------------------------------------------------------------------------------
// Decoder forward for one tile.  E,G -> H1 -> H2 -> H3 -> heads -> OUT rows (10 x TP).
// H3 is written to `H3buf` (the H1 rows in forward-only kernels, a separate buffer in backward).
// SDF_ONLY skips the colour head (rgb outputs are written as 0).
// ------------------------------------------------------------------------------------------
template <bool SDF_ONLY>
__device__ __forceinline__ void mlp_forward_tile(const float* __restrict__ prep, float* sm, float* H3buf) {
    const int tid = threadIdx.x, tx = tid & 15, m0 = (tid >> 4) * 4;
    float* E = sm + ROW_E * LDA; float* G = sm + ROW_G * LDA;
    float* H1 = sm + ROW_H1 * LDA; float* H2 = sm + ROW_H2 * LDA;
    float* PS = sm + ROW_SM * LDA; float* OUT = sm + ROW_OUT * LDA;
    float acc[4][8];
    // pts_linear.0 + ReLU  (51 -> 128)
    init_bias(acc, prep + OFF_B1, tx);
    gemm_fwd_acc<D_EP>(acc, E, prep + PREP_F1, tx, m0);
    store_acc<true>(acc, H1, tx, m0);
    __syncthreads();
    // pts_linear.2  (128 -> 128), no activation
    init_bias(acc, prep + OFF_B2, tx);
    gemm_fwd_acc<D_H>(acc, H1, prep + PREP_F2, tx, m0);
    store_acc<false>(acc, H2, tx, m0);
    __syncthreads();
    // sdf_linear.0 + ReLU on [sdf_emb = h[:64], grid(32)]  (96 -> 128)
    init_bias(acc, prep + OFF_BS1, tx);
    gemm_fwd_acc<D_SDF_EMB>(acc, H2, prep + PREP_F3, tx, m0);
    gemm_fwd_acc<D_GRID>(acc, G, prep + PREP_F3 + D_SDF_EMB * 128, tx, m0);
    store_acc<true>(acc, H3buf, tx, m0);       // H1 is dead after layer 2 in forward-only kernels
    __syncthreads();
    // heads: thread (m, part) accumulates a quarter of each dot product
    const int m = tid & (TP - 1), part = tid >> 6;
    {
        float s[N_CLASS] = {0.f, 0.f, 0.f, 0.f, 0.f};
        const float* ws2 = prep + OFF_WS2;
#pragma unroll 4
        for (int kk = 0; kk < 32; ++kk) {
            const int k = part * 32 + kk;
            const float h = H3buf[k * LDA + m];
#pragma unroll
            for (int c = 0; c < N_CLASS; ++c) s[c] = fmaf(__ldg(ws2 + c * D_H + k), h, s[c]);
        }
#pragma unroll
        for (int c = 0; c < N_CLASS; ++c) PS[(part * 8 + c) * LDA + m] = s[c];
        float r[3] = {0.f, 0.f, 0.f};
        if (!SDF_ONLY) {
            const float* wr = prep + OFF_WR;
#pragma unroll 4
            for (int kk = 0; kk < 16; ++kk) {
                const int k = part * 16 + kk;
                const float h = H2[(D_SDF_EMB + k) * LDA + m];
#pragma unroll
                for (int c = 0; c < 3; ++c) r[c] = fmaf(__ldg(wr + c * D_RGB_IN + k), h, r[c]);
            }
            const int j1 = min(part * 13 + 13, D_E);
            for (int j = part * 13; j < j1; ++j) {
                const float e = E[j * LDA + m];
#pragma unroll
                for (int c = 0; c < 3; ++c) r[c] = fmaf(__ldg(wr + c * D_RGB_IN + 64 + j), e, r[c]);
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) PS[(part * 8 + 5 + c) * LDA + m] = r[c];
    }
    __syncthreads();
    if (part == 0) {
        float zl[N_CLASS], rgb[3];
#pragma unroll
        for (int c = 0; c < N_CLASS; ++c)
            zl[c] = __ldg(prep + OFF_BS2 + c) + ((PS[c * LDA + m] + PS[(8 + c) * LDA + m]) + (PS[(16 + c) * LDA + m] + PS[(24 + c) * LDA + m]));
#pragma unroll
        for (int c = 0; c < 3; ++c)
            rgb[c] = SDF_ONLY ? 0.f
                              : __ldg(prep + OFF_BR + c) + ((PS[(5 + c) * LDA + m] + PS[(13 + c) * LDA + m]) + (PS[(21 + c) * LDA + m] + PS[(29 + c) * LDA + m]));
        float mx = zl[0];
#pragma unroll
        for (int c = 1; c < N_CLASS; ++c) mx = fmaxf(mx, zl[c]);
        float p[N_CLASS], se = 0.f;
#pragma unroll
        for (int c = 0; c < N_CLASS; ++c) { p[c] = expf(zl[c] - mx); se += p[c]; }
        float ent = 0.f, ex = 0.f;
#pragma unroll
        for (int c = 0; c < N_CLASS; ++c) {
            p[c] = p[c] / se;
            ent += p[c] * log2f(p[c] + 1e-5f);
            ex += p[c] * (float)c;
        }
        OUT[0 * LDA + m] = rgb[0]; OUT[1 * LDA + m] = rgb[1]; OUT[2 * LDA + m] = rgb[2];
        OUT[3 * LDA + m] = (ex / 4.0f - 0.5f) * 2.0f;            // model/decoder.py:72
        OUT[4 * LDA + m] = -1.0f * ent;                          // model/decoder.py:68
#pragma unroll
        for (int c = 0; c < N_CLASS; ++c) OUT[(5 + c) * LDA + m] = p[c];
    }
}

// Coalesced store of a tile's outputs OUT[c][m] (row length ld, tp points per tile) to raw (N,10).
__device__ __forceinline__ void store_raw_tile(const float* OUT, int ld, int tp, float* __restrict__ raw, int64_t tile, int64_t N,
                                               int tid, int nthreads) {
    const int64_t base = tile * tp;
    const int nv = (int)min((int64_t)tp, N - base);
    for (int idx = tid; idx < nv * MF_RAW_DIM; idx += nthreads) {
        const int m = idx / MF_RAW_DIM, c = idx % MF_RAW_DIM;
        raw[base * MF_RAW_DIM + idx] = OUT[c * ld + m];
    }
}
