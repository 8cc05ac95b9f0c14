// Kernels + C-ABI entry points of the neural-field query path:
//   mf_hashgrid_*, mf_freq_*, mf_mlp_*, mf_field_query(_bwd), mf_field_query_rays(_bwd).
#include "field_bwd.cuh"
#include "field_launch.cuh"
#include "field_tc_launch.cuh"
#include "field_tc_bwd.cuh"
#include "field_tc_bwd2.cuh"
#include "field_tc_bwd3.cuh"

// ---------------------------------------------------------------------------------------------
// Weight re-layout (runs once per optimiser step; 36.6 k floats).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mlp_prepare_simt(const float* __restrict__ mlp, float* __restrict__ prep, int i) {
    if (i >= PREP_SIMT_SIZE) return;
    float v = 0.f;
    if (i < MF_MLP_PARAMS) {
        v = mlp[i];
    } else if (i >= PREP_F1) {
        int r;
        if (i < PREP_B1) {            // forward copies: F[k][tx][i8] = W[n = tx + 16 i8][k]
            int off, K, Kreal;
            if (i < PREP_F2) { r = i - PREP_F1; off = OFF_W1; K = D_E; Kreal = D_E; }
            else if (i < PREP_F3) { r = i - PREP_F2; off = OFF_W2; K = D_H; Kreal = D_H; }
            else { r = i - PREP_F3; off = OFF_WS1; K = D_SDF_IN; Kreal = D_SDF_IN; }
            const int k = r >> 7, tx = (r >> 3) & 15, i8 = r & 7;
            const int n = tx + 16 * i8;
            v = (k < Kreal) ? mlp[off + n * K + k] : 0.f;
        } else {                      // backward copies: B[n][tx][i] = W[n][k = tx + 16 i]
            int off, K, KI;
            if (i < PREP_B2) { r = i - PREP_B1; off = OFF_W1; K = D_E; KI = 4; }
            else if (i < PREP_B3) { r = i - PREP_B2; off = OFF_W2; K = D_H; KI = 8; }
            else { r = i - PREP_B3; off = OFF_WS1; K = D_SDF_IN; KI = 6; }
            const int n = r / (16 * KI), rem = r % (16 * KI), tx = rem / KI, ii = rem % KI;
            const int k = tx + 16 * ii;
            v = (k < K) ? mlp[off + n * K + k] : 0.f;
        }
    }
    prep[i] = v;
}

// bf16 hi/lo, 128B-swizzled K-major weight image + fp32 head section for the tcgen05 decoder (field_tc.cuh)
__device__ __forceinline__ void mlp_prepare_tc(const float* __restrict__ mlp, uint8_t* __restrict__ img, int t) {
    // one thread per (layer, n, k) weight element: 128 x (64 + 128 + 128)
    if (t < 128 * 320) {
        const int n = t / 320, kk = t % 320;
        float w; int hi_off, lo_off, k;
        if (kk < 64) {                     // pts_linear.0, slot order
            k = kk; const int e = tc_e_slot_to_index(k);
            w = e >= 0 ? mlp[OFF_W1 + n * D_E + e] : 0.f;
            hi_off = IMG_W1_HI; lo_off = IMG_W1_LO;
        } else if (kk < 192) {             // pts_linear.2
            k = kk - 64; w = mlp[OFF_W2 + n * D_H + k];
            hi_off = IMG_W2_HI; lo_off = IMG_W2_LO;
        } else {                           // sdf_linear.0 (K = 96, zero padded to 128)
            k = kk - 192; w = k < D_SDF_IN ? mlp[OFF_WS1 + n * D_SDF_IN + k] : 0.f;
            hi_off = IMG_W3_HI; lo_off = IMG_W3_LO;
        }
        const __nv_bfloat16 h = __float2bfloat16_rn(w);
        const __nv_bfloat16 l = __float2bfloat16_rn(w - __bfloat162float(h));
        const uint32_t off = (uint32_t)(k >> 6) * IMG_BLOCK + sw128_offset(n, k & 63);
        *reinterpret_cast<__nv_bfloat16*>(img + hi_off + off) = h;
        *reinterpret_cast<__nv_bfloat16*>(img + lo_off + off) = l;
    } else if (t < 128 * 320 + F_COUNT) {
        const int j = t - 128 * 320;
        float v = 0.f;
        if (j < F_B2) v = mlp[OFF_B1 + j];
        else if (j < F_BS1) v = mlp[OFF_B2 + (j - F_B2)];
        else if (j < F_WR_EMB) v = mlp[OFF_BS1 + (j - F_BS1)];
        else if (j < F_WR_E) { const int c = (j - F_WR_EMB) / 64, k = (j - F_WR_EMB) % 64; v = mlp[OFF_WR + c * D_RGB_IN + k]; }
        else if (j < F_BR) {
            const int c = (j - F_WR_E) / 64, e = tc_e_slot_to_index((j - F_WR_E) % 64);
            v = e >= 0 ? mlp[OFF_WR + c * D_RGB_IN + 64 + e] : 0.f;
        }
        else if (j < F_WS2) v = (j - F_BR) < 3 ? mlp[OFF_BR + (j - F_BR)] : 0.f;
        else if (j < F_BS2) v = mlp[OFF_WS2 + (j - F_WS2)];
        else v = (j - F_BS2) < 5 ? mlp[OFF_BS2 + (j - F_BS2)] : 0.f;
        reinterpret_cast<float*>(img + IMG_F32)[j] = v;
    }
}

// one launch for both layouts: the first blocks write the fp32 copies, the rest the tensor-core image
constexpr int PREP_BLOCKS_SIMT = (PREP_SIMT_SIZE + 255) / 256;
constexpr int PREP_BLOCKS_TC = (128 * 320 + F_COUNT + 255) / 256;
__global__ void __launch_bounds__(256) mlp_prepare_kernel(const float* __restrict__ mlp, float* __restrict__ prep) {
    if (blockIdx.x < PREP_BLOCKS_SIMT) mlp_prepare_simt(mlp, prep, blockIdx.x * 256 + threadIdx.x);
    else mlp_prepare_tc(mlp, reinterpret_cast<uint8_t*>(prep + PREP_TC), (blockIdx.x - PREP_BLOCKS_SIMT) * 256 + threadIdx.x);
}

// (the generic forward kernel templates live in field_launch.cuh / field_tc_launch.cuh)
__global__ void __launch_bounds__(NT, 2) mlp_fwd_kernel(const float* embed, const float* embed_pos, const float* pts,
                                                        const float* __restrict__ prep, float* __restrict__ out, int64_t N) {
    extern __shared__ __align__(16) float sm[];
    const int64_t n_tiles = (N + TP - 1) / TP;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        load_features_tile(embed, embed_pos, pts, tile, N, sm);
        __syncthreads();
        mlp_forward_tile<false>(prep, sm, sm + ROW_H1 * LDA);
        __syncthreads();
        store_raw_tile(sm + ROW_OUT * LDA, LDA, TP, out, tile, N, threadIdx.x, NT);
        __syncthreads();
    }
}

// ---------------------------------------------------------------------------------------------
// Backward kernels.  part: [gridDim.x][MF_MLP_PARAMS] per-CTA partial parameter gradients.
// ---------------------------------------------------------------------------------------------
template <class Src, bool WANT_DX>
__global__ void __launch_bounds__(NT, 1) field_bwd_kernel(FieldDev f, Src src, const float* __restrict__ d_raw,
                                                          float* __restrict__ grad_grid, float* __restrict__ part,
                                                          float* __restrict__ d_pts, int64_t N_all, ActiveMap am) {
    extern __shared__ __align__(16) float sm[];
    float* gpart = part + (size_t)blockIdx.x * MF_MLP_PARAMS;
    for (int i = threadIdx.x; i < MF_MLP_PARAMS; i += NT) gpart[i] = 0.f;
    __syncthreads();
    const int64_t N = am.n(N_all);                     // active points only
    const int64_t n_tiles = (N + TP - 1) / TP;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        encode_tile(f, src, tile, N, sm, am);
        __syncthreads();
        mlp_forward_tile<false>(f.prep, sm, sm + ROW_H3 * LDA);
        __syncthreads();
        head_backward_tile(d_raw, tile, N, sm, am);
        __syncthreads();
        mlp_backward_tile<WANT_DX>(f.prep, sm, gpart);
        encode_backward_tile<Src, WANT_DX>(f, src, tile, N, sm, grad_grid, d_pts, am);
        __syncthreads();
    }
}

// Input gradients only on the fp32 decoder (no weight gradients, no grid scatter): the pose gradients of the overlap-region
// SDF consistency (overlap_kernels.cu), whose residual is a small difference of two fields and needs the fp32 recomputation.
// Every point's d_pts depends on that point and its d_raw row alone (no atomics): deterministic.
template <class Src>
__global__ void __launch_bounds__(NT, 1) field_bwd_dx_kernel(FieldDev f, Src src, const float* __restrict__ d_raw,
                                                             float* __restrict__ d_pts, int64_t N_all, ActiveMap am) {
    extern __shared__ __align__(16) float sm[];
    const int64_t N = am.n(N_all);
    const int64_t n_tiles = (N + TP - 1) / TP;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        encode_tile(f, src, tile, N, sm, am);
        __syncthreads();
        mlp_forward_tile<false>(f.prep, sm, sm + ROW_H3 * LDA);
        __syncthreads();
        head_backward_tile(d_raw, tile, N, sm, am);
        __syncthreads();
        mlp_backward_tile<true, false>(f.prep, sm, nullptr);
        encode_backward_tile<Src, true, false>(f, src, tile, N, sm, nullptr, d_pts, am);
        __syncthreads();
    }
}

template <bool WANT_DX>
__global__ void __launch_bounds__(NT, 1) mlp_bwd_kernel(const float* embed, const float* embed_pos, const float* pts,
                                                        const float* __restrict__ prep, const float* __restrict__ d_out,
                                                        float* __restrict__ part, float* __restrict__ d_embed,
                                                        float* __restrict__ d_embed_pos, float* __restrict__ d_pts, int64_t N) {
    extern __shared__ __align__(16) float sm[];
    float* gpart = part + (size_t)blockIdx.x * MF_MLP_PARAMS;
    for (int i = threadIdx.x; i < MF_MLP_PARAMS; i += NT) gpart[i] = 0.f;
    __syncthreads();
    const int64_t n_tiles = (N + TP - 1) / TP;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        load_features_tile(embed, embed_pos, pts, tile, N, sm);
        __syncthreads();
        mlp_forward_tile<false>(prep, sm, sm + ROW_H3 * LDA);
        __syncthreads();
        head_backward_tile(d_out, tile, N, sm);
        __syncthreads();
        mlp_backward_tile<WANT_DX>(prep, sm, gpart);
        const float* E = sm + ROW_E * LDA; const float* G = sm + ROW_G * LDA;
        const int64_t base = tile * TP;
        const int nv = (int)min((int64_t)TP, N - base);
        if (d_embed)
            for (int idx = threadIdx.x; idx < nv * D_GRID; idx += NT)
                d_embed[base * D_GRID + idx] = G[(idx % D_GRID) * LDA + idx / D_GRID];
        if (WANT_DX) {
            if (d_embed_pos)
                for (int idx = threadIdx.x; idx < nv * D_FREQ; idx += NT)
                    d_embed_pos[base * D_FREQ + idx] = E[(3 + idx % D_FREQ) * LDA + idx / D_FREQ];
            if (d_pts)
                for (int idx = threadIdx.x; idx < nv * 3; idx += NT) d_pts[base * 3 + idx] = E[(idx % 3) * LDA + idx / 3];
        }
        __syncthreads();
    }
}

// grad_mlp[dst(s)] += sum over CTAs of part[cta][s].  A block covers 32 consecutive partial entries s; warp j sums the
// CTAs j, j+8, ... in order (coalesced 128-byte reads), then the 8 partial sums are combined in a fixed order ->
// deterministic.  transposed != 0: the three 128-row weight matrices are stored [in][out] inside each partial
// (tensor-core path) and dst() undoes that.
// transposed == 2 (role-split tensor-core backward): additionally, the LAST block forms the gradient of pts_linear.2.bias, which
// that kernel does not accumulate per point because it is linear in two other bias gradients of the same call:
//   dH[p][n] = sum_m dZ3[p][m] Ws1[m][n] (n < 64),  dH[p][n] = sum_c dRGB[p][c] Wr[c][n - 64] (n >= 64)
//   =>  db2[n] = sum_m dbs1[m] Ws1[m][n]  resp.  sum_c dbr[c] Wr[c][n - 64];      mlp = the state_dict-ordered weight blob.
__global__ void __launch_bounds__(256) reduce_partials_kernel(const float* __restrict__ part, int n_cta, float* __restrict__ grad_mlp,
                                                              int transposed, const float* __restrict__ mlp) {
    __shared__ float acc[8][32];
    if (transposed == 2 && blockIdx.x == gridDim.x - 1) {
        __shared__ float dbs1[D_H], dbr[4];
        const int t = threadIdx.x;
        if (t < D_H + 3) {
            const int sidx = t < D_H ? OFF_BS1 + t : OFF_BR + (t - D_H);
            float s = 0.f;
            for (int c = 0; c < n_cta; ++c) s += __ldg(&part[(size_t)c * MF_MLP_PARAMS + sidx]);
            if (t < D_H) dbs1[t] = s; else dbr[t - D_H] = s;
        }
        __syncthreads();
        if (t < D_H) {
            float s = 0.f;
            if (t < D_SDF_EMB) {
                for (int m = 0; m < D_H; ++m) s = fmaf(dbs1[m], __ldg(&mlp[OFF_WS1 + m * D_SDF_IN + t]), s);
            } else {
                for (int c = 0; c < 3; ++c) s = fmaf(dbr[c], __ldg(&mlp[OFF_WR + c * D_RGB_IN + (t - D_SDF_EMB)]), s);
            }
            grad_mlp[OFF_B2 + t] += s;
        }
        return;
    }
    const int lane = threadIdx.x & 31, j = threadIdx.x >> 5;
    const int sidx = blockIdx.x * 32 + lane;
    const bool on = sidx < MF_MLP_PARAMS;
    float s = 0.f;
    if (on) {
#pragma unroll 4
        for (int c = j; c < n_cta; c += 8) s += __ldg(&part[(size_t)c * MF_MLP_PARAMS + sidx]);
    }
    acc[j][lane] = s;
    __syncthreads();
    const bool b2_entry = transposed == 2 && sidx >= OFF_B2 && sidx < OFF_B2 + D_H;      // owned by the last block
    if (j == 0 && on && !b2_entry) {
        const float tot = ((acc[0][lane] + acc[1][lane]) + (acc[2][lane] + acc[3][lane])) + ((acc[4][lane] + acc[5][lane]) + (acc[6][lane] + acc[7][lane]));
        int dst = sidx;
        if (transposed) {
            if (sidx < OFF_B1) { const int r = sidx - OFF_W1; dst = OFF_W1 + (r % D_H) * D_E + r / D_H; }
            else if (sidx >= OFF_W2 && sidx < OFF_B2) { const int r = sidx - OFF_W2; dst = OFF_W2 + (r % D_H) * D_H + r / D_H; }
            else if (sidx >= OFF_WS1 && sidx < OFF_BS1) { const int r = sidx - OFF_WS1; dst = OFF_WS1 + (r % D_H) * D_SDF_IN + r / D_H; }
        }
        grad_mlp[dst] += tot;
    }
}

// d_rays_o[r] = sum_s d_pts[r,s]; d_rays_d[r] = sum_s z[r,s] d_pts[r,s]   (warp per ray, fixed order)
__global__ void ray_grad_reduce_kernel(const float* __restrict__ d_pts, const float* __restrict__ z,
                                       float* __restrict__ d_o, float* __restrict__ d_d, int64_t R, int S) {
    const int64_t r = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    float so[3] = {0.f, 0.f, 0.f}, sd[3] = {0.f, 0.f, 0.f};
    for (int s = lane; s < S; s += 32) {
        const float zz = z[r * S + s];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const float g = d_pts[(r * S + s) * 3 + k];
            so[k] += g; sd[k] = fmaf(zz, g, sd[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) { so[k] = warp_sum(so[k]); sd[k] = warp_sum(sd[k]); }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 3; ++k) { d_o[r * 3 + k] = so[k]; d_d[r * 3 + k] = sd[k]; }
    }
}

// ---------------------------------------------------------------------------------------------
// Stand-alone encodings (drop-in tcnn.Encoding replacements).
// ---------------------------------------------------------------------------------------------
__global__ void hashgrid_fwd_kernel(FieldDev f, const float* __restrict__ x, float* __restrict__ out,
                                    uint32_t* __restrict__ idx_dump, int64_t N) {
    // thread per (point, level); level fastest so that the 32 outputs of a point are written contiguously
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int L = f.n_levels;
    if (t >= N * L) return;
    const int64_t i = t / L; const int l = (int)(t % L);
    const float xv[3] = {x[i * 3], x[i * 3 + 1], x[i * 3 + 2]};
    uint32_t idx[8];
    const float2 v = grid_level_fwd(xv, reinterpret_cast<const float2*>(f.grid), level_info(f, l), idx);
    reinterpret_cast<float2*>(out)[t] = v;
    if (idx_dump) {
#pragma unroll
        for (int c = 0; c < 8; ++c) idx_dump[t * 8 + c] = idx[c];
    }
}

template <bool WANT_DX>
__global__ void hashgrid_bwd_kernel(FieldDev f, const float* __restrict__ x, const float* __restrict__ dy,
                                    float* __restrict__ grad, float* __restrict__ dx_out, int64_t N) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int L = f.n_levels;                       // 16 levels -> the 16 lanes of a half warp share a point
    const bool active = t < N * L;
    const int64_t i = active ? t / L : 0; const int l = (int)(t % L);
    float dx[3] = {0.f, 0.f, 0.f};
    if (active) {
        const float xv[3] = {x[i * 3], x[i * 3 + 1], x[i * 3 + 2]};
        const float2 g = reinterpret_cast<const float2*>(dy)[t];
        grid_level_bwd<WANT_DX>(xv, g, reinterpret_cast<const float2*>(f.grid), grad, level_info(f, l), dx);
    }
    if (WANT_DX) {
#pragma unroll
        for (int d = 0; d < 3; ++d)
#pragma unroll
            for (int o = 8; o > 0; o >>= 1) dx[d] += __shfl_xor_sync(0xffffffffu, dx[d], o);
        if (active && l == 0) { dx_out[i * 3] = dx[0]; dx_out[i * 3 + 1] = dx[1]; dx_out[i * 3 + 2] = dx[2]; }
    }
}

__global__ void freq_fwd_kernel(const float* __restrict__ x, float* __restrict__ out, int D, int K, int64_t N) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int W = D * K * 2;
    if (t >= N * W) return;
    const int64_t i = t / W; const int j = (int)(t % W);
    const int d = j / (2 * K), k = (j / 2) % K, s = j & 1;
    out[t] = sinf(freq_arg(x[i * D + d], k, s));
}

__global__ void freq_bwd_kernel(const float* __restrict__ x, const float* __restrict__ dy, float* __restrict__ dx,
                                int D, int K, int64_t N) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= N * D) return;
    const int64_t i = t / D; const int d = (int)(t % D);
    const float xv = x[t];
    float s = 0.f;
    for (int k = 0; k < K; ++k)
        for (int ph = 0; ph < 2; ++ph)
            s += dy[i * (D * K * 2) + d * 2 * K + 2 * k + ph] * cosf(freq_arg(xv, k, ph)) * ldexpf(3.14159274101257324f, k);
    dx[t] = s;
}

// ---------------------------------------------------------------------------------------------
// Host side
// ---------------------------------------------------------------------------------------------
int mf_field_to_dev(const mf_field* f, FieldDev* d) {
    if (!f || !f->grid || !f->mlp_prep) { mf_set_error("mf_field: null grid/mlp_prep"); return MF_ERR_INVALID; }
    if (f->meta.n_levels != 16 || f->meta.n_features != 2) {
        mf_set_error("fused field kernels are built for 16 levels x 2 features (got %d x %d)", f->meta.n_levels, f->meta.n_features);
        return MF_ERR_UNSUPPORTED;
    }
    d->grid = f->grid; d->prep = f->mlp_prep; d->feat = nullptr;
    d->tc_img = reinterpret_cast<const uint8_t*>(f->mlp_prep + PREP_TC);
    for (int k = 0; k < 3; ++k) { d->na[k] = f->norm_a[k]; d->nb[k] = f->norm_b[k]; }
    d->nf = f->norm_factor;
    for (int l = 0; l < f->meta.n_levels; ++l)
        if (f->meta.offset[l] & 1u) { mf_set_error("mf_field: level offsets must be even (16-byte reductions)"); return MF_ERR_INVALID; }
    d->impl = f->decoder_impl == 0 ? mf_decoder_impl() : (f->decoder_impl == 1 ? 1 : 0);
    d->n_levels = f->meta.n_levels;
    for (int l = 0; l < MF_MAX_LEVELS; ++l) {
        d->scale[l] = f->meta.scale[l]; d->res[l] = f->meta.resolution[l]; d->size[l] = f->meta.size[l];
        d->offset[l] = f->meta.offset[l]; d->hashed[l] = f->meta.hashed[l];
    }
    return MF_OK;
}

static int meta_to_dev(const mf_grid_meta* m, const float* grid, FieldDev* d) {
    if (!m || m->n_levels < 1 || m->n_levels > MF_MAX_LEVELS || m->n_features != 2) {
        mf_set_error("hash grid: need 1..16 levels and 2 features per level");
        return MF_ERR_UNSUPPORTED;
    }
    memset(d, 0, sizeof(*d));
    d->grid = grid; d->n_levels = m->n_levels; d->nf = 1.0;
    for (int l = 0; l < m->n_levels; ++l) {
        d->scale[l] = m->scale[l]; d->res[l] = m->resolution[l]; d->size[l] = m->size[l];
        d->offset[l] = m->offset[l]; d->hashed[l] = m->hashed[l];
    }
    return MF_OK;
}

MF_API int mf_hashgrid_meta(int log2_T, int n_levels, int n_features, int base_res, double per_level_scale, mf_grid_meta* m) {
    MF_CHECK_ARG(m != nullptr);
    MF_CHECK_ARG(n_levels >= 1 && n_levels <= MF_MAX_LEVELS);
    MF_CHECK_ARG(log2_T >= 1 && log2_T <= 30);
    memset(m, 0, sizeof(*m));
    m->n_levels = n_levels; m->n_features = n_features; m->log2_hashmap_size = log2_T; m->base_resolution = base_res;
    // tcnn: per_level_scale is read from JSON as float; log2 taken in float.  exp2f is taken as the
    // correctly rounded fp32 value (oracle/hashgrid.py explains why this is fixed normatively).
    const float log2_pls = log2f((float)per_level_scale);
    uint32_t off = 0;
    for (int l = 0; l < n_levels; ++l) {
        const float arg = (float)l * log2_pls;
        const float s = (float)exp2((double)arg) * (float)base_res - 1.0f;
        const uint32_t r = (uint32_t)ceilf(s) + 1u;
        const uint32_t max_params = UINT32_MAX / 2;
        uint32_t n = (powf((float)r, 3.0f) > (float)max_params) ? max_params : r * r * r;
        n = (n + 7u) / 8u * 8u;
        const uint32_t cap = 1u << log2_T;
        if (n > cap) n = cap;
        // grid_index(): the dense stride loop stops once stride > size; hashed iff size < final stride
        uint32_t stride = 1;
        for (int d = 0; d < 3 && stride <= n; ++d) stride *= r;
        m->scale[l] = s; m->resolution[l] = r; m->size[l] = n; m->offset[l] = off; m->hashed[l] = (n < stride) ? 1u : 0u;
        off += n;
    }
    m->offset[n_levels] = off;
    return MF_OK;
}

MF_API int mf_hashgrid_fwd(const float* x, const float* grid, const mf_grid_meta* meta, float* out, uint32_t* idx_dump,
                           int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(x && grid && out);
    FieldDev d; int rc = meta_to_dev(meta, grid, &d); if (rc) return rc;
    const int64_t T = N * d.n_levels;
    hashgrid_fwd_kernel<<<(unsigned)((T + 255) / 256), 256, 0, (cudaStream_t)stream>>>(d, x, out, idx_dump, N);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_hashgrid_bwd(const float* x, const float* dL_dy, const float* grid, const mf_grid_meta* meta,
                           float* grad_grid, float* dL_dx, int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(x && dL_dy && grid && grad_grid);
    MF_CHECK_ARG(((uintptr_t)grad_grid & 15) == 0);          // the scatter uses 16-byte reductions
    FieldDev d; int rc = meta_to_dev(meta, grid, &d); if (rc) return rc;
    for (int l = 0; l < d.n_levels; ++l) MF_CHECK_ARG((d.offset[l] & 1u) == 0);
    if (dL_dx && d.n_levels != 16) { mf_set_error("mf_hashgrid_bwd: input gradient needs 16 levels"); return MF_ERR_UNSUPPORTED; }
    const int64_t T = N * d.n_levels;
    const unsigned blocks = (unsigned)((T + 255) / 256);
    if (dL_dx) hashgrid_bwd_kernel<true><<<blocks, 256, 0, (cudaStream_t)stream>>>(d, x, dL_dy, grad_grid, dL_dx, N);
    else hashgrid_bwd_kernel<false><<<blocks, 256, 0, (cudaStream_t)stream>>>(d, x, dL_dy, grad_grid, nullptr, N);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_freq_fwd(const float* x, float* out, int n_dims, int n_frequencies, int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0 && n_dims > 0 && n_frequencies > 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(x && out);
    const int64_t T = N * n_dims * n_frequencies * 2;
    freq_fwd_kernel<<<(unsigned)((T + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, out, n_dims, n_frequencies, N);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_freq_bwd(const float* x, const float* dL_dy, float* dL_dx, int n_dims, int n_frequencies, int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0 && n_dims > 0 && n_frequencies > 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(x && dL_dy && dL_dx);
    const int64_t T = N * n_dims;
    freq_bwd_kernel<<<(unsigned)((T + 255) / 256), 256, 0, (cudaStream_t)stream>>>(x, dL_dy, dL_dx, n_dims, n_frequencies, N);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int64_t mf_mlp_prep_size(void) { return PREP_SIZE; }

MF_API int mf_mlp_prepare(const float* mlp, float* mlp_prep, void* stream) {
    MF_CHECK_ARG(mlp && mlp_prep);
    mlp_prepare_kernel<<<PREP_BLOCKS_SIMT + PREP_BLOCKS_TC, 256, 0, (cudaStream_t)stream>>>(mlp, mlp_prep);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int64_t mf_mlp_grad_workspace_size(void) { return (int64_t)mf_sm_count_cached() * MF_MLP_PARAMS; }

MF_API int mf_mlp_fwd(const float* embed, const float* embed_pos, const float* pts, const float* mlp_prep, float* out,
                      int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(embed && embed_pos && pts && mlp_prep && out);
    int rc = set_smem(mlp_fwd_kernel, SMEM_FWD); if (rc) return rc;
    mlp_fwd_kernel<<<persistent_grid(N, 2), NT, SMEM_FWD, (cudaStream_t)stream>>>(embed, embed_pos, pts, mlp_prep, out, N);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_mlp_bwd(const float* embed, const float* embed_pos, const float* pts, const float* mlp_prep,
                      const float* d_out, float* grad_mlp, float* d_embed, float* d_embed_pos, float* d_pts,
                      float* workspace, int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(embed && embed_pos && pts && mlp_prep && d_out && grad_mlp && workspace);
    const bool want_dx = d_embed_pos || d_pts;
    const int grid = persistent_grid(N, 1);
    cudaStream_t st = (cudaStream_t)stream;
    if (want_dx) {
        int rc = set_smem(mlp_bwd_kernel<true>, SMEM_BWD); if (rc) return rc;
        mlp_bwd_kernel<true><<<grid, NT, SMEM_BWD, st>>>(embed, embed_pos, pts, mlp_prep, d_out, workspace, d_embed, d_embed_pos, d_pts, N);
    } else {
        int rc = set_smem(mlp_bwd_kernel<false>, SMEM_BWD); if (rc) return rc;
        mlp_bwd_kernel<false><<<grid, NT, SMEM_BWD, st>>>(embed, embed_pos, pts, mlp_prep, d_out, workspace, d_embed, nullptr, nullptr, N);
    }
    MF_LAUNCH_CHECK();
    reduce_partials_kernel<<<(MF_MLP_PARAMS + 31) / 32, 256, 0, st>>>(workspace, grid, grad_mlp, 0, nullptr);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Active-point compaction.  A point whose upstream gradient row d_raw[i][0..9] is all zero (a sample behind the
// surface: no loss term sees it, helper_functions/utils.py:21-47) adds exactly zero to every gradient, so the
// backward kernels skip it.  Ordered (ascending point index => run-to-run deterministic tiles), two small kernels:
// flags + per-block counts, then every block sums the counts before it and writes its ranks.
// ---------------------------------------------------------------------------------------------
constexpr int ACT_BLK = 1024;

__global__ void __launch_bounds__(ACT_BLK) active_count_kernel(const float* __restrict__ d_raw, int64_t N,
                                                               uint32_t* __restrict__ flags, int* __restrict__ blk_cnt) {
    const int64_t i = (int64_t)blockIdx.x * ACT_BLK + threadIdx.x;
    bool on = false;
    if (i < N) {
        const float2* g = reinterpret_cast<const float2*>(d_raw + i * MF_RAW_DIM);      // 40-byte rows: 8-byte aligned
#pragma unroll
        for (int k = 0; k < MF_RAW_DIM / 2; ++k) { const float2 v = __ldg(g + k); on |= (v.x != 0.f) | (v.y != 0.f); }
    }
    const uint32_t word = __ballot_sync(0xffffffffu, on);
    if ((threadIdx.x & 31) == 0) flags[i >> 5] = word;
    const int total = __syncthreads_count(on);
    if (threadIdx.x == 0) blk_cnt[blockIdx.x] = total;
}

__global__ void __launch_bounds__(ACT_BLK) active_fill_kernel(const uint32_t* __restrict__ flags, const int* __restrict__ blk_cnt,
                                                              int* __restrict__ idx, int* __restrict__ n_active) {
    __shared__ int wsum[32];
    __shared__ int base_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    int part = 0;
    for (int j = tid; j < (int)blockIdx.x; j += ACT_BLK) part += blk_cnt[j];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if (lane == 0) wsum[warp] = part;
    __syncthreads();
    if (warp == 0) {
        int v = wsum[lane];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (lane == 0) base_s = v;
    }
    __syncthreads();
    const int base = base_s;
    const int64_t i = (int64_t)blockIdx.x * ACT_BLK + tid;
    const uint32_t word = flags[i >> 5];                      // the flag array is padded to whole blocks
    __syncthreads();
    if (lane == 0) wsum[warp] = __popc(word);
    __syncthreads();
    if (warp == 0) {                                          // exclusive scan of the 32 warp counts
        const int c = wsum[lane];
        int v = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int t = __shfl_up_sync(0xffffffffu, v, o); if (lane >= o) v += t; }
        wsum[lane] = v - c;
        if (lane == 31 && blockIdx.x == gridDim.x - 1) *n_active = base + v;
    }
    __syncthreads();
    if ((word >> lane) & 1u) idx[base + wsum[warp] + __popc(word & ((1u << lane) - 1u))] = (int)i;
}

static inline int64_t act_blocks(int64_t N) { return (N + ACT_BLK - 1) / ACT_BLK; }
// scratch (in 4-byte words) behind the partials / point gradients: idx[N] | flags[blocks * 32] | blk_cnt[blocks] | count
static inline int64_t act_scratch_words(int64_t N) { return N + act_blocks(N) * 33 + 4; }

static int compact_active_points(const float* d_raw, int64_t N, float* scratch, ActiveMap* am, cudaStream_t st) {
    if ((uintptr_t)d_raw & 7) { mf_set_error("backward: the upstream gradient must be 8-byte aligned"); return MF_ERR_INVALID; }
    if (N >= (int64_t)1 << 31) { mf_set_error("backward: more than 2^31 points"); return MF_ERR_INVALID; }
    const int64_t nb = act_blocks(N);
    int* idx = reinterpret_cast<int*>(scratch);
    uint32_t* flags = reinterpret_cast<uint32_t*>(idx + N);
    int* blk_cnt = reinterpret_cast<int*>(flags + nb * 32);
    int* count = blk_cnt + nb;
    active_count_kernel<<<(unsigned)nb, ACT_BLK, 0, st>>>(d_raw, N, flags, blk_cnt);
    MF_LAUNCH_CHECK();
    active_fill_kernel<<<(unsigned)nb, ACT_BLK, 0, st>>>(flags, blk_cnt, idx, count);
    MF_LAUNCH_CHECK();
    am->idx = idx; am->count = count;
    return MF_OK;
}

// ... followed by the CTA-private scratch of the role-split tensor-core backward (parked activations, field_tc_bwd2.cuh)
static inline int64_t cta_scratch_words() { return (int64_t)mf_sm_count_cached() * b2::SCR_CTA_WORDS; }

MF_API int64_t mf_field_bwd_workspace_size(int64_t n_points, int want_point_grads) {
    if (n_points < 0) n_points = 0;
    return mf_mlp_grad_workspace_size() + (want_point_grads ? 3 * n_points : 0) + act_scratch_words(n_points) + cta_scratch_words();
}

template <class Src>
static int launch_field_bwd(const FieldDev& d, const Src& src, const float* d_raw, float* grad_grid, float* grad_mlp,
                            float* d_pts, float* workspace, float* scratch, int64_t N, cudaStream_t st) {
    // workspace: per-CTA partials; scratch: act_scratch_words(N) words for the active-point list
    ActiveMap am{nullptr, nullptr};
    int rc0 = compact_active_points(d_raw, N, scratch, &am, st); if (rc0) return rc0;
    if (d_pts) MF_CUDA(cudaMemsetAsync(d_pts, 0, (size_t)N * 3 * sizeof(float), st));   // skipped points: exactly zero
    const bool params = grad_grid != nullptr;          // false: input gradients only (pose refinement, overlap consistency)
    if (!params && !d_pts) {
        mf_set_error("backward without parameter gradients needs a ray / point gradient output");
        return MF_ERR_INVALID;
    }
    if (!params && d.impl == 1) {
        const int grid = persistent_grid(N, 1);
        int rc = set_smem(field_bwd_dx_kernel<Src>, SMEM_BWD); if (rc) return rc;
        field_bwd_dx_kernel<Src><<<grid, NT, SMEM_BWD, st>>>(d, src, d_raw, d_pts, N, am);
        MF_LAUNCH_CHECK();
        return MF_OK;
    }
    if (d.impl != 1) {                                 // tcgen05 path: 128-point tiles, one CTA per SM
        const int64_t tiles = (N + TC_TP - 1) / TC_TP;
        const int64_t cap = mf_sm_count_cached();
        const int grid = (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
        mf_ktimer_begin(1, st);
        if (!params) {
            int rc = set_smem(field_bwd_tc_kernel<Src, true, false>, SMEM_TC_BWD); if (rc) return rc;
            field_bwd_tc_kernel<Src, true, false><<<grid, TC_NT, SMEM_TC_BWD, st>>>(d, src, d_raw, nullptr, nullptr, d_pts, N, am, mf_tc_error_flag(), mf_tc_profile_buffer());
            mf_ktimer_end(1, st);
            MF_LAUNCH_CHECK();
            return MF_OK;
        }
        if (!d_pts && mf_bwd_impl() != 1) {                // role-split kernels (parameter gradients only)
            uint32_t* cta_scr = reinterpret_cast<uint32_t*>(scratch + act_scratch_words(N));
            if (mf_bwd_impl() == 3 && d.feat) {            // four roles (A/B only: measured slower, field_tc_bwd3.cuh); needs the feature cache
                int rc = set_smem(field_bwd_tc3_kernel<Src>, b3::SMEM); if (rc) return rc;
                field_bwd_tc3_kernel<Src><<<grid, b3::B3_NT, b3::SMEM, st>>>(d, src, d_raw, grad_grid, workspace, cta_scr, N, am, mf_tc_error_flag(), mf_tc_profile_buffer());
            } else {                                       // three roles (default)
                int rc = set_smem(field_bwd_tc2_kernel<Src>, b2::SMEM); if (rc) return rc;
                field_bwd_tc2_kernel<Src><<<grid, b2::B2_NT, b2::SMEM, st>>>(d, src, d_raw, grad_grid, workspace, cta_scr, N, am, mf_tc_error_flag(), mf_tc_profile_buffer(),
                                                                             mf_bwd_impl() == 2 ? 0 : 1);
            }
            mf_ktimer_end(1, st);
            MF_LAUNCH_CHECK();
            reduce_partials_kernel<<<(MF_MLP_PARAMS + 31) / 32 + 1, 256, 0, st>>>(workspace, grid, grad_mlp, 2, d.prep);
            MF_LAUNCH_CHECK();
            return MF_OK;
        }
        if (d_pts) {
            int rc = set_smem(field_bwd_tc_kernel<Src, true>, SMEM_TC_BWD); if (rc) return rc;
            field_bwd_tc_kernel<Src, true><<<grid, TC_NT, SMEM_TC_BWD, st>>>(d, src, d_raw, grad_grid, workspace, d_pts, N, am, mf_tc_error_flag(), mf_tc_profile_buffer());
        } else {
            int rc = set_smem(field_bwd_tc_kernel<Src, false>, SMEM_TC_BWD); if (rc) return rc;
            field_bwd_tc_kernel<Src, false><<<grid, TC_NT, SMEM_TC_BWD, st>>>(d, src, d_raw, grad_grid, workspace, nullptr, N, am, mf_tc_error_flag(), mf_tc_profile_buffer());
        }
        mf_ktimer_end(1, st);
        MF_LAUNCH_CHECK();
        reduce_partials_kernel<<<(MF_MLP_PARAMS + 31) / 32, 256, 0, st>>>(workspace, grid, grad_mlp, 1, nullptr);
        MF_LAUNCH_CHECK();
        return MF_OK;
    }
    const int grid = persistent_grid(N, 1);
    if (d_pts) {
        int rc = set_smem(field_bwd_kernel<Src, true>, SMEM_BWD); if (rc) return rc;
        field_bwd_kernel<Src, true><<<grid, NT, SMEM_BWD, st>>>(d, src, d_raw, grad_grid, workspace, d_pts, N, am);
    } else {
        int rc = set_smem(field_bwd_kernel<Src, false>, SMEM_BWD); if (rc) return rc;
        field_bwd_kernel<Src, false><<<grid, NT, SMEM_BWD, st>>>(d, src, d_raw, grad_grid, workspace, nullptr, N, am);
    }
    MF_LAUNCH_CHECK();
    reduce_partials_kernel<<<(MF_MLP_PARAMS + 31) / 32, 256, 0, st>>>(workspace, grid, grad_mlp, 0, nullptr);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_field_query(const float* pts, const mf_field* field, int normalize, float* out, int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(pts && out);
    FieldDev d; int rc = mf_field_to_dev(field, &d); if (rc) return rc;
    SrcPoints src{pts, normalize};
    return launch_field_fwd_auto<SrcPoints, EpiRaw, false>(d, src, EpiRaw{out}, N, (cudaStream_t)stream);
}

MF_API int mf_field_query_bwd(const float* pts, const mf_field* field, int normalize, const float* d_out, float* grad_grid,
                              float* grad_mlp, float* d_pts, float* workspace, int64_t N, void* stream) {
    MF_CHECK_ARG(N >= 0);
    if (N == 0) return MF_OK;
    MF_CHECK_ARG(pts && d_out && workspace);
    MF_CHECK_ARG((grad_grid == nullptr) == (grad_mlp == nullptr));      // both NULL: point gradients only (needs d_pts)
    MF_CHECK_ARG(grad_grid || d_pts);
    MF_CHECK_ARG(((uintptr_t)grad_grid & 15) == 0);          // the scatter uses 16-byte reductions
    FieldDev d; int rc = mf_field_to_dev(field, &d); if (rc) return rc;
    SrcPoints src{pts, normalize};
    return launch_field_bwd(d, src, d_out, grad_grid, grad_mlp, d_pts, workspace, workspace + mf_mlp_grad_workspace_size(), N,
                            (cudaStream_t)stream);
}

MF_API int64_t mf_feat_cache_size(int64_t n_points) {
    return ((n_points + TC_TP - 1) / TC_TP) * (int64_t)FEAT_TILE_WORDS * 4;
}

MF_API int mf_field_query_rays(const float* rays_o, const float* rays_d, const float* z, const mf_field* field, float* raw,
                               void* feat, int64_t R, int S, void* stream) {
    MF_CHECK_ARG(R >= 0 && S > 0);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(rays_o && rays_d && z && raw);
    FieldDev d; int rc = mf_field_to_dev(field, &d); if (rc) return rc;
    d.feat = (uint32_t*)feat;
    SrcRays src{rays_o, rays_d, z, S};
    return launch_field_fwd_auto<SrcRays, EpiRaw, false>(d, src, EpiRaw{raw}, R * S, (cudaStream_t)stream, nullptr, false, 0);
}

MF_API int mf_field_query_rays_bwd(const float* rays_o, const float* rays_d, const float* z, const mf_field* field,
                                   const float* d_raw, const void* feat, float* grad_grid, float* grad_mlp, float* d_rays_o,
                                   float* d_rays_d, float* workspace, int64_t R, int S, void* stream) {
    MF_CHECK_ARG(R >= 0 && S > 0);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(rays_o && rays_d && z && d_raw && workspace);
    MF_CHECK_ARG((grad_grid == nullptr) == (grad_mlp == nullptr));      // both NULL: ray gradients only (needs d_rays_o / d_rays_d)
    MF_CHECK_ARG(((uintptr_t)grad_grid & 15) == 0);          // the scatter uses 16-byte reductions
    MF_CHECK_ARG((d_rays_o == nullptr) == (d_rays_d == nullptr));
    FieldDev d; int rc = mf_field_to_dev(field, &d); if (rc) return rc;
    d.feat = (uint32_t*)feat;
    SrcRays src{rays_o, rays_d, z, S};
    cudaStream_t st = (cudaStream_t)stream;
    // the per-point dL/dp buffer lives behind the per-CTA partials in the workspace
    float* d_pts = d_rays_o ? workspace + mf_mlp_grad_workspace_size() : nullptr;
    float* scratch = workspace + mf_mlp_grad_workspace_size() + (d_rays_o ? 3 * R * S : 0);
    rc = launch_field_bwd(d, src, d_raw, grad_grid, grad_mlp, d_pts, workspace, scratch, R * S, st);
    if (rc) return rc;
    if (d_rays_o) {
        ray_grad_reduce_kernel<<<(unsigned)((R + 7) / 8), 256, 0, st>>>(d_pts, z, d_rays_o, d_rays_d, R, S);
        MF_LAUNCH_CHECK();
    }
    return MF_OK;
}
