// Backward of the fused field evaluation for one tile (recompute-forward, then back-propagate).
// See field_core.cuh for the forward and the shared-memory map.
#pragma once
#include "field_core.cuh"

// Head backward for point m (threads 0..TP-1): d_raw (10) + forward OUT rows -> DZ rows
// (dlogits 0..4, drgb_raw 5..7).   model/decoder.py:65-74 differentiated.
__device__ __forceinline__ void head_backward_tile(const float* __restrict__ d_raw, int64_t tile, int64_t N, float* sm,
                                                   const ActiveMap am = ActiveMap{nullptr, nullptr}) {
    const int m = threadIdx.x;
    if (m >= TP) return;
    const float* OUT = sm + ROW_OUT * LDA;
    float* DZ = sm + ROW_DZ * LDA;
    const int64_t slot = tile * TP + m;
    const int64_t i = slot < N ? am(slot) : 0;
    float g[MF_RAW_DIM];
#pragma unroll
    for (int c = 0; c < MF_RAW_DIM; ++c) g[c] = (slot < N) ? d_raw[i * MF_RAW_DIM + c] : 0.f;
    float p[N_CLASS], dp[N_CLASS], dot = 0.f;
#pragma unroll
    for (int c = 0; c < N_CLASS; ++c) {
        p[c] = OUT[(5 + c) * LDA + m];
        // sdf = sum p_c c / 2 - 1 ; entropy = -sum p log2(p + 1e-5)
        const float q = p[c] + 1e-5f;
        dp[c] = g[5 + c] + g[3] * (0.5f * (float)c) - g[4] * (log2f(q) + p[c] / (q * 0.6931471805599453f));
        dot = fmaf(p[c], dp[c], dot);
    }
#pragma unroll
    for (int c = 0; c < N_CLASS; ++c) DZ[c * LDA + m] = p[c] * (dp[c] - dot);
#pragma unroll
    for (int c = 0; c < 3; ++c) DZ[(5 + c) * LDA + m] = g[c];
}

// Full decoder backward for one tile.  On entry: E, G, H1, H2, H3, OUT hold the forward
// activations and DZ the head gradients.  On exit: G rows hold dL/dgrid-features, and (WANT_DX)
// E rows hold dL/de.  gpart is this CTA's private partial of the parameter gradient blob.
// PARAMS = false (with WANT_DX): input gradients only, no weight or bias gradients (gpart unused).
template <bool WANT_DX, bool PARAMS = true>
__device__ __forceinline__ void mlp_backward_tile(const float* __restrict__ prep, float* sm, float* __restrict__ gpart) {
    const int tid = threadIdx.x, tx = tid & 15, m0 = (tid >> 4) * 4;
    float* E = sm + ROW_E * LDA; float* G = sm + ROW_G * LDA;
    float* H1 = sm + ROW_H1 * LDA; float* H2 = sm + ROW_H2 * LDA; float* H3 = sm + ROW_H3 * LDA;
    float* DZ = sm + ROW_DZ * LDA;

    // ---- weight gradients of the two small heads -------------------------------------------------
    if (PARAMS) {   // sdf_linear.2: dW[c][k] += sum_m DZ[c][m] H3[k][m]   (5 x 128): thread (k = tid & 127, half)
        const int k = tid & 127, half = tid >> 7;
        const int c0 = half ? 3 : 0, c1 = half ? 5 : 3;
        float s[3] = {0.f, 0.f, 0.f};
        for (int m = 0; m < TP; m += 4) {
            const float4 h = *reinterpret_cast<const float4*>(H3 + k * LDA + m);
            for (int c = c0; c < c1; ++c) {
                const float4 z = *reinterpret_cast<const float4*>(DZ + c * LDA + m);
                s[c - c0] += (z.x * h.x + z.y * h.y) + (z.z * h.z + z.w * h.w);
            }
        }
        for (int c = c0; c < c1; ++c) gpart[OFF_WS2 + c * D_H + k] += s[c - c0];
        // rgb_linear.0: dW[c][j] += sum_m DZ[5+c][m] X[j][m], X = [H2[64..127], E[0..50]]  (3 x 115)
        if (k < D_RGB_IN) {
            const float* xrow = (k < 64) ? (H2 + (D_SDF_EMB + k) * LDA) : (E + (k - 64) * LDA);
            const int r0 = half ? 2 : 0, r1 = half ? 3 : 2;
            float t[2] = {0.f, 0.f};
            for (int m = 0; m < TP; m += 4) {
                const float4 h = *reinterpret_cast<const float4*>(xrow + m);
                for (int c = r0; c < r1; ++c) {
                    const float4 z = *reinterpret_cast<const float4*>(DZ + (5 + c) * LDA + m);
                    t[c - r0] += (z.x * h.x + z.y * h.y) + (z.z * h.z + z.w * h.w);
                }
            }
            for (int c = r0; c < r1; ++c) gpart[OFF_WR + c * D_RGB_IN + k] += t[c - r0];
        }
        // biases of both heads: warp w < 8 reduces DZ row w
        const int w = tid >> 5, lane = tid & 31;
        float b = DZ[w * LDA + lane] + DZ[w * LDA + lane + 32];
        b = warp_sum(b);
        if (lane == 0) gpart[(w < 5 ? OFF_BS2 + w : OFF_BR + (w - 5))] += b;
    }
    __syncthreads();

    // ---- dZ3 = (Ws2^T dlogits) * relu'(H3) in place of H3; d rgb_emb into H2[64..127] ------------
    {
        const float* ws2 = prep + OFF_WS2;
        const float* wr = prep + OFF_WR;
        for (int idx = tid; idx < D_H * TP; idx += NT) {
            const int m = idx & (TP - 1), k = idx >> 6;
            float s = 0.f;
#pragma unroll
            for (int c = 0; c < N_CLASS; ++c) s = fmaf(__ldg(ws2 + c * D_H + k), DZ[c * LDA + m], s);
            const float h = H3[k * LDA + m];
            H3[k * LDA + m] = h > 0.f ? s : 0.f;
            if (k < 64) {
                float r = 0.f;
#pragma unroll
                for (int c = 0; c < 3; ++c) r = fmaf(__ldg(wr + c * D_RGB_IN + k), DZ[(5 + c) * LDA + m], r);
                H2[(D_SDF_EMB + k) * LDA + m] = r;
            }
        }
    }
    __syncthreads();

    // ---- sdf_linear.0: wgrad (128 x 96) on A3 = [H2[0..63], G], bias ------------------------------
    if (PARAMS) {
        wgrad_tile<6>(H3, [&](int k) -> const float* { return k < 64 ? H2 + k * LDA : G + (k - 64) * LDA; }, D_SDF_IN,
                      gpart + OFF_WS1, tid);
        bias_grad_tile(H3, gpart + OFF_BS1, tid);
    }
    {   // dgrad: dA3[k][m] = sum_n Ws1[n][k] dZ3[n][m], k < 96 (registers; written after the barrier)
        float acc[4][6];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int i = 0; i < 6; ++i) acc[mi][i] = 0.f;
        gemm_dgrad_acc<6>(acc, H3, prep + PREP_B3, tx, m0);
        __syncthreads();                                   // wgrad above has finished reading H2[0..63] and G
#pragma unroll
        for (int i = 0; i < 6; ++i) {
            const int k = tx + 16 * i;
            float* dst = (k < 64) ? (H2 + k * LDA) : (G + (k - 64) * LDA);
            *reinterpret_cast<float4*>(dst + m0) = make_float4(acc[0][i], acc[1][i], acc[2][i], acc[3][i]);
        }
    }
    __syncthreads();

    // ---- pts_linear.2: wgrad (128 x 128) with dH = H2, A = H1; dgrad -> dZ1 in place of H1 -------
    if (PARAMS) {
        wgrad_tile<8>(H2, [&](int k) -> const float* { return H1 + k * LDA; }, D_H, gpart + OFF_W2, tid);
        bias_grad_tile(H2, gpart + OFF_B2, tid);
    }
    {
        float acc[4][8];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int i = 0; i < 8; ++i) acc[mi][i] = 0.f;
        gemm_dgrad_acc<8>(acc, H2, prep + PREP_B2, tx, m0);
        __syncthreads();                                   // wgrad above has finished reading H1
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float* row = H1 + (tx + 16 * i) * LDA + m0;
            const float4 h = *reinterpret_cast<const float4*>(row);
            *reinterpret_cast<float4*>(row) = make_float4(h.x > 0.f ? acc[0][i] : 0.f, h.y > 0.f ? acc[1][i] : 0.f,
                                                          h.z > 0.f ? acc[2][i] : 0.f, h.w > 0.f ? acc[3][i] : 0.f);
        }
    }
    __syncthreads();

    // ---- pts_linear.0: wgrad (128 x 51) with dZ1 = H1, A = E; optional dgrad -> dE ----------------
    if (PARAMS) {
        wgrad_tile<4>(H1, [&](int k) -> const float* { return E + k * LDA; }, D_E, gpart + OFF_W1, tid);
        bias_grad_tile(H1, gpart + OFF_B1, tid);
    }
    if (WANT_DX) {
        float acc[4][4];
#pragma unroll
        for (int mi = 0; mi < 4; ++mi)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[mi][i] = 0.f;
        gemm_dgrad_acc<4>(acc, H1, prep + PREP_B1, tx, m0);
        __syncthreads();                                   // wgrad above has finished reading E
        const float* wr = prep + OFF_WR;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int k = tx + 16 * i;
            if (k < D_E) {
                float v[4] = {acc[0][i], acc[1][i], acc[2][i], acc[3][i]};
#pragma unroll
                for (int c = 0; c < 3; ++c) {             // colour head reads e directly (model/decoder.py:61)
                    const float wv = __ldg(wr + c * D_RGB_IN + 64 + k);
                    const float4 z = *reinterpret_cast<const float4*>(DZ + (5 + c) * LDA + m0);
                    v[0] = fmaf(wv, z.x, v[0]); v[1] = fmaf(wv, z.y, v[1]); v[2] = fmaf(wv, z.z, v[2]); v[3] = fmaf(wv, z.w, v[3]);
                }
                *reinterpret_cast<float4*>(E + k * LDA + m0) = make_float4(v[0], v[1], v[2], v[3]);
            }
        }
    }
    __syncthreads();
}

// Encoder backward: scatter dL/dgrid-features (G rows) into grad_grid and, if WANT_DX, gather
// dL/dx from the grid levels, the frequency features and the raw xyz input; the four partial
// sums per point are combined through the PS rows and converted to dL/dp by the source.
// PARAMS = false: no scatter into grad_grid (input gradients only).
template <class Src, bool WANT_DX, bool PARAMS = true>
__device__ __forceinline__ void encode_backward_tile(const FieldDev& f, const Src& src, int64_t tile, int64_t N,
                                                     float* sm, float* __restrict__ grad_grid,
                                                     float* __restrict__ d_pts,
                                                     const ActiveMap am = ActiveMap{nullptr, nullptr}) {
    const int tid = threadIdx.x, m = tid & (TP - 1), q = tid >> 6;
    const int64_t slot = tile * TP + m;
    const bool valid = slot < N;
    const int64_t i = valid ? am(slot) : 0;
    float* E = sm + ROW_E * LDA; float* G = sm + ROW_G * LDA; float* PS = sm + ROW_SM * LDA;
    float x[3] = {0.f, 0.f, 0.f};
    if (valid) src.point(i, f, x);
    float dx[3] = {0.f, 0.f, 0.f};
    const float2* grid2 = reinterpret_cast<const float2*>(f.grid);
    if (valid) {
#pragma unroll
        for (int ll = 0; ll < 4; ++ll) {
            const int l = q * 4 + ll;
            const float2 dy = make_float2(G[(2 * l) * LDA + m], G[(2 * l + 1) * LDA + m]);
            grid_level_bwd<WANT_DX, PARAMS>(x, dy, grid2, grad_grid, level_info(f, l), dx);
        }
    }
    if (WANT_DX) {
#pragma unroll
        for (int jj = 0; jj < 12; ++jj) {
            const int j = q * 12 + jj, d = j >> 4, k = (j & 15) >> 1, s = j & 1;
            // d sin(arg)/dx = 2^k * PI * cos(arg)
            const float de = E[(3 + j) * LDA + m];
            const float c = cosf(freq_arg(x[d], k, s)) * ldexpf(3.14159274101257324f, k) * de;
            if (d == 0) dx[0] += c; else if (d == 1) dx[1] += c; else dx[2] += c;
        }
        if (q == 0) { dx[0] += E[0 * LDA + m]; dx[1] += E[1 * LDA + m]; dx[2] += E[2 * LDA + m]; }
        PS[(q * 4 + 0) * LDA + m] = dx[0]; PS[(q * 4 + 1) * LDA + m] = dx[1]; PS[(q * 4 + 2) * LDA + m] = dx[2];
        __syncthreads();
        if (q == 0 && valid) {
            float t[3], dp[3];
#pragma unroll
            for (int d = 0; d < 3; ++d)
                t[d] = (PS[d * LDA + m] + PS[(4 + d) * LDA + m]) + (PS[(8 + d) * LDA + m] + PS[(12 + d) * LDA + m]);
            src.dx_to_dp(f, t, dp);
            d_pts[i * 3 + 0] = dp[0]; d_pts[i * 3 + 1] = dp[1]; d_pts[i * 3 + 2] = dp[2];
        }
    }
}
