// Depth sampling along rays, SDF->weight volume rendering, the rgb/depth/sdf/free-space losses
// (forward and backward) and ray generation.
// Reference: model/scene_rep.py:58-103,157-176,190-238; helper_functions/utils.py:21-111;
// mipsfusion.py:320-322; helper_functions/geometry_helper.py:107-123.
#include <limits.h>

#include "mf_common.cuh"

constexpr int MAX_S = 128;     // samples per ray handled by one warp (4 per lane)

struct RenderCfgDev {
    int n_u, n_r, perturb, rgb_missing_nz;
    float tr;          // fp32(trunc): "sdf / trunc" with a python scalar
    float sctr;        // fp32(sc_factor * trunc): "z_min + sc_factor * trunc"
    float T;           // fp32(trunc * sc_factor): truncation of the losses
    float twoT;        // fp32(2 * truncation)
    float depth_trunc;
    float emd_w;
    int ld_rgb, ld_d;  // row strides (floats) of target_rgb / target_d: 3 / 1 for contiguous tensors, 10 / 10 for column slices of
                       // the reference loop's (R,10) batch tensor (mipsfusion.py:316-322), which then need no copy
};

static RenderCfgDev cfg_to_dev(const mf_render_cfg* c) {
    RenderCfgDev d;
    d.n_u = c->n_samples_d; d.n_r = c->n_range_d; d.perturb = c->perturb; d.rgb_missing_nz = c->rgb_missing_nz;
    d.tr = (float)c->trunc; d.sctr = (float)(c->sc_factor * c->trunc);
    const double T = c->trunc * c->sc_factor;
    d.T = (float)T; d.twoT = (float)(2.0 * T);
    d.depth_trunc = (float)c->depth_trunc; d.emd_w = (float)c->emd_w;
    d.ld_rgb = 3; d.ld_d = 1;
    return d;
}

// ---------------------------------------------------------------------------------------------
// z sampling: one block per ray.  Merge of the uniform list and the around-depth list by rank,
// stratified jitter, and the global front / sdf mask counts.
// ---------------------------------------------------------------------------------------------
__global__ void sample_z_kernel(const float* __restrict__ target_d, const float* __restrict__ u,
                                const float* __restrict__ lin_u, const float* __restrict__ lin_r,
                                const float* __restrict__ lin_fb, RenderCfgDev c, float* __restrict__ z,
                                unsigned long long* __restrict__ counts, int64_t R) {
    extern __shared__ float zs[];
    __shared__ int cnt[2];
    mf_pdl_wait(); mf_pdl_trigger();
    const int64_t r = blockIdx.x;
    const int S = c.n_u + c.n_r;
    const bool has_d = target_d != nullptr;
    const float d = has_d ? target_d[r * c.ld_d] : 0.f;
    const bool around = d > 0.f;                      // rows with target_d <= 0 fall back to linspace(near, far)
    if (threadIdx.x < 2) cnt[threadIdx.x] = 0;
    for (int e = threadIdx.x; e < S; e += blockDim.x) {
        float v; int rank;
        if (e < c.n_u) {
            v = lin_u[e]; rank = e;
            for (int k = 0; k < c.n_r; ++k) {
                const float sv = around ? __fadd_rn(lin_r[k], d) : lin_fb[k];
                rank += (sv < v);
            }
        } else {
            const int k = e - c.n_u;
            v = around ? __fadd_rn(lin_r[k], d) : lin_fb[k];
            rank = k;
            for (int i = 0; i < c.n_u; ++i) rank += (lin_u[i] <= v);
        }
        zs[rank] = v;
    }
    __syncthreads();
    int n_front = 0, n_sdf = 0;
    for (int j = threadIdx.x; j < S; j += blockDim.x) {
        float zj = zs[j];
        if (c.perturb && u) {
            const float lower = (j == 0) ? zs[0] : 0.5f * __fadd_rn(zs[j], zs[j - 1]);
            const float upper = (j == S - 1) ? zs[S - 1] : 0.5f * __fadd_rn(zs[j + 1], zs[j]);
            zj = __fadd_rn(lower, __fmul_rn(__fsub_rn(upper, lower), u[r * S + j]));
        }
        z[r * S + j] = zj;
        if (has_d) {
            const bool front = zj < __fsub_rn(d, c.T);
            const bool back = zj > __fadd_rn(d, c.T);
            n_front += front;
            n_sdf += (!front && !back && d > 0.f);
        }
    }
    if (has_d) {
        for (int o = 16; o > 0; o >>= 1) {
            n_front += __shfl_xor_sync(0xffffffffu, n_front, o);
            n_sdf += __shfl_xor_sync(0xffffffffu, n_sdf, o);
        }
        if ((threadIdx.x & 31) == 0) { atomicAdd(&cnt[0], n_front); atomicAdd(&cnt[1], n_sdf); }
        __syncthreads();
        if (threadIdx.x == 0) {
            atomicAdd(&counts[0], (unsigned long long)cnt[0]);
            atomicAdd(&counts[1], (unsigned long long)cnt[1]);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Per-ray quantities shared by the forward and backward render kernels (one warp per ray).
// ---------------------------------------------------------------------------------------------
struct RaySamples {
    float sdf[4], z[4], sig[4], wt[4];    // wt = masked, un-normalised weight
    bool in[4];
    int inds; float wsum;
};

__device__ __forceinline__ void load_ray(const float* __restrict__ raw, const float* __restrict__ z, int64_t r, int S,
                                         int lane, const RenderCfgDev& c, RaySamples& q) {
    int cand = INT_MAX;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int s = lane + 32 * t;
        q.in[t] = s < S;
        q.sdf[t] = q.in[t] ? raw[(r * S + s) * MF_RAW_DIM + 3] : 0.f;
        q.z[t] = q.in[t] ? z[r * S + s] : 0.f;
        if (s < S - 1) {
            const float nxt = raw[(r * S + s + 1) * MF_RAW_DIM + 3];
            if (__fmul_rn(nxt, q.sdf[t]) < 0.f) cand = min(cand, s);        // scene_rep.py:70-72
        }
    }
    cand = warp_min_i(cand);
    q.inds = (cand == INT_MAX) ? 0 : cand;
    const float z_min = z[r * S + q.inds];
    const float thr = __fadd_rn(z_min, c.sctr);                             // scene_rep.py:75
    float ws = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const float xs = __fdiv_rn(q.sdf[t], c.tr);
        q.sig[t] = sigmoidf_(xs);
        const float w = q.sig[t] * sigmoidf_(-xs);                          // scene_rep.py:68
        q.wt[t] = (q.in[t] && q.z[t] < thr) ? w : 0.f;
        ws += q.wt[t];
    }
    q.wsum = warp_sum(ws);
}

__global__ void __launch_bounds__(256) render_loss_fwd_kernel(
    const float* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ target_rgb,
    const float* __restrict__ target_d, RenderCfgDev c, float* __restrict__ out_rgb, float* __restrict__ out_depth,
    float* __restrict__ out_aux, float* __restrict__ out_w, int32_t* __restrict__ inds, float* __restrict__ scratch,
    int64_t R, int S) {
    mf_pdl_wait(); mf_pdl_trigger();
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    RaySamples q;
    load_ray(raw, z, r, S, lane, c, q);
    const float inv = 1.0f / (q.wsum + 1e-8f);
    float rgb[3] = {0.f, 0.f, 0.f}, depth = 0.f, acc = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (!q.in[t]) continue;
        const int s = lane + 32 * t;
        const float w = q.wt[t] * inv;
        if (out_w) out_w[r * S + s] = w;
        const float* rw = raw + (r * S + s) * MF_RAW_DIM;
#pragma unroll
        for (int k = 0; k < 3; ++k) rgb[k] = fmaf(w, sigmoidf_(rw[k]), rgb[k]);
        depth = fmaf(w, q.z[t], depth);
        acc += w;
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) rgb[k] = warp_sum(rgb[k]);
    depth = warp_sum(depth); acc = warp_sum(acc);
    float var = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const float dz = q.z[t] - depth;
        var = fmaf(q.wt[t] * inv, dz * dz, var);
    }
    var = warp_sum(var);
    if (lane == 0) {
        out_rgb[r * 3] = rgb[0]; out_rgb[r * 3 + 1] = rgb[1]; out_rgb[r * 3 + 2] = rgb[2];
        out_depth[r] = depth;
        if (out_aux) {
            out_aux[r * 3] = var;
            out_aux[r * 3 + 1] = 1.0f / fmaxf(1e-10f, depth / acc);          // scene_rep.py:100
            out_aux[r * 3 + 2] = acc;
        }
        if (inds) inds[r] = q.inds;
    }
    if (!target_d) return;
    // ---- loss partial sums of this ray (helper_functions/utils.py:71-111, scene_rep.py:211-226) ----
    const float d = target_d[r * c.ld_d];
    const bool valid = d > 0.f && d < c.depth_trunc;
    const float mk = (valid || c.rgb_missing_nz) ? 1.f : 0.f;
    float fs2 = 0.f, sdf2 = 0.f, fs1 = 0.f, sdf1 = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (!q.in[t]) continue;
        const int s = lane + 32 * t;
        const float zz = q.z[t], sd = q.sdf[t];
        const bool front = zz < __fsub_rn(d, c.T);
        const bool back = zz > __fadd_rn(d, c.T);
        const float fm = front ? 1.f : 0.f;
        const float sm_ = (!front && !back && d > 0.f) ? 1.f : 0.f;
        const float e1 = sd * fm - fm;
        fs2 = fmaf(e1, e1, fs2);
        const float e2 = (zz + sd * c.T) * sm_ - d * sm_;
        sdf2 = fmaf(e2, e2, sdf2);
        if (c.emd_w > 0.f) {
            const float* p = raw + (r * S + s) * MF_RAW_DIM + 5;
            const float gt = __fdiv_rn(__fadd_rn(__fsub_rn(d, zz), c.T), c.twoT) * 4.0f;
            float a = 0.f, b = 0.f;
#pragma unroll
            for (int k = 0; k < 5; ++k) { a = fmaf(p[k], (float)(4 - k), a); b = fmaf(fabsf(gt - (float)k), p[k], b); }
            fs1 = fmaf(a, fm, fs1);
            sdf1 = fmaf(b, sm_, sdf1);
        }
    }
    fs2 = warp_sum(fs2); sdf2 = warp_sum(sdf2); fs1 = warp_sum(fs1); sdf1 = warp_sum(sdf1);
    if (lane == 0) {
        float rs = 0.f;
        if (target_rgb)
#pragma unroll
            for (int k = 0; k < 3; ++k) { const float e = rgb[k] * mk - target_rgb[r * c.ld_rgb + k] * mk; rs = fmaf(e, e, rs); }
        float* sc = scratch + r * 8;
        sc[0] = rs; sc[1] = valid ? (depth - d) * (depth - d) : 0.f; sc[2] = valid ? 1.f : 0.f;
        sc[3] = fs2; sc[4] = sdf2; sc[5] = fs1; sc[6] = sdf1; sc[7] = 0.f;
    }
}

// Fixed-order fp64 reduction of the per-ray partial sums and the final loss scalars.
__global__ void __launch_bounds__(1024) loss_finalize_kernel(const float* __restrict__ scratch,
                                                             const unsigned long long* __restrict__ counts,
                                                             RenderCfgDev c, float* __restrict__ losses, int64_t R, int S) {
    __shared__ double red[32][8];
    mf_pdl_wait(); mf_pdl_trigger();
    double s[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    const float4* rows = reinterpret_cast<const float4*>(scratch);            // 8 floats per ray: two 16-byte loads
    for (int64_t r = threadIdx.x; r < R; r += 1024) {
        const float4 a = rows[2 * r], b = rows[2 * r + 1];
        s[0] += (double)a.x; s[1] += (double)a.y; s[2] += (double)a.z; s[3] += (double)a.w;
        s[4] += (double)b.x; s[5] += (double)b.y; s[6] += (double)b.z;
    }
#pragma unroll
    for (int k = 0; k < 7; ++k) s[k] = warp_sum_d(s[k]);
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0)
#pragma unroll
        for (int k = 0; k < 7; ++k) red[w][k] = s[k];
    __syncthreads();
    if (w != 0) return;
    double t[7];
#pragma unroll
    for (int k = 0; k < 7; ++k) t[k] = warp_sum_d(red[lane][k]);              // the 32 warp sums: a second fixed-order tree
    if (threadIdx.x == 0) {
        const double RS = (double)R * (double)S;
        const float n_fs = (float)counts[0], n_sdf = (float)counts[1];
        const float n = (float)(counts[0] + counts[1]);
        const float fs_w = 1.0f - n_fs / n, sdf_w = 1.0f - n_sdf / n;      // utils.py:45-47
        const float rgb_loss = (float)(t[0] / (3.0 * (double)R));
        const float depth_loss = (float)(t[1] / t[2]);                      // NaN when no valid ray, as the reference
        float fs_loss = (float)(t[3] / RS) * fs_w, sdf_loss = (float)(t[4] / RS) * sdf_w;
        if (c.emd_w > 0.f) {
            fs_loss += (float)(t[5] / RS) / 250.0f * c.emd_w;
            sdf_loss += (float)(t[6] / RS) / 5000.0f * c.emd_w;
        }
        losses[0] = rgb_loss; losses[1] = depth_loss; losses[2] = sdf_loss; losses[3] = fs_loss;
        losses[4] = -10.0f * logf(rgb_loss) / logf(10.0f);                  // mse2psnr, utils.py:5-6
        losses[5] = fs_w; losses[6] = sdf_w; losses[7] = (float)t[2];
    }
}

struct LossGrads { const float* p[4]; };     // upstream gradients of rgb / depth / sdf / fs loss, each a device scalar or NULL (= 0)

__global__ void __launch_bounds__(256) render_loss_bwd_kernel(
    const float* __restrict__ raw, const float* __restrict__ z, const float* __restrict__ target_rgb,
    const float* __restrict__ target_d, const float* __restrict__ losses, RenderCfgDev c,
    LossGrads g_losses, const float* __restrict__ g_rgb, const float* __restrict__ g_depth,
    float* __restrict__ d_raw, int64_t R, int S) {
    mf_pdl_wait(); mf_pdl_trigger();
    const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (r >= R) return;
    RaySamples q;
    load_ray(raw, z, r, S, lane, c, q);
    const float inv = 1.0f / (q.wsum + 1e-8f);
    // recompute the rendered colour / depth of this ray
    float sg[4][3];
    float rgb[3] = {0.f, 0.f, 0.f}, depth = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        const int s = lane + 32 * t;
        const float w = q.wt[t] * inv;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            sg[t][k] = q.in[t] ? sigmoidf_(raw[(r * S + s) * MF_RAW_DIM + k]) : 0.f;
            rgb[k] = fmaf(w, sg[t][k], rgb[k]);
        }
        depth = fmaf(w, q.z[t], depth);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) rgb[k] = warp_sum(rgb[k]);
    depth = warp_sum(depth);
    // upstream gradients of the rendered maps
    const bool has_t = target_d != nullptr;
    const float d = has_t ? target_d[r * c.ld_d] : 0.f;
    const bool valid = has_t && d > 0.f && d < c.depth_trunc;
    const float mk = (valid || c.rgb_missing_nz) ? 1.f : 0.f;
    const float gl_rgb = g_losses.p[0] ? __ldg(g_losses.p[0]) : 0.f, gl_depth = g_losses.p[1] ? __ldg(g_losses.p[1]) : 0.f;
    const float gl_sdf = g_losses.p[2] ? __ldg(g_losses.p[2]) : 0.f, gl_fs = g_losses.p[3] ? __ldg(g_losses.p[3]) : 0.f;
    float G_rgb[3], G_depth = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        G_rgb[k] = g_rgb ? g_rgb[r * 3 + k] : 0.f;
        if (has_t && target_rgb) G_rgb[k] += gl_rgb * 2.0f * mk * (rgb[k] * mk - target_rgb[r * c.ld_rgb + k] * mk) / (3.0f * (float)R);
    }
    if (g_depth) G_depth = g_depth[r];
    if (valid && gl_depth != 0.f) G_depth += gl_depth * 2.0f * (depth - d) / losses[7];
    float a[4], abar = 0.f;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        a[t] = G_rgb[0] * sg[t][0] + G_rgb[1] * sg[t][1] + G_rgb[2] * sg[t][2] + G_depth * q.z[t];
        abar = fmaf(q.wt[t] * inv, a[t], abar);
    }
    abar = warp_sum(abar);
    const float fs_w = has_t ? losses[5] : 0.f, sdf_w = has_t ? losses[6] : 0.f;
    const float invRS = 1.0f / ((float)R * (float)S);
#pragma unroll
    for (int t = 0; t < 4; ++t) {
        if (!q.in[t]) continue;
        const int s = lane + 32 * t;
        const float zz = q.z[t], sd = q.sdf[t], sgm = q.sig[t];
        float* o = d_raw + (r * S + s) * MF_RAW_DIM;
        // through the normalised weights (the mask and the sign-change index carry no gradient)
        float dsdf = 0.f;
        if (q.wt[t] != 0.f) dsdf = (a[t] - abar) * inv * (sgm * (1.0f - sgm) * (1.0f - 2.0f * sgm)) / c.tr;
        float dp[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        if (has_t) {
            const bool front = zz < __fsub_rn(d, c.T);
            const bool back = zz > __fadd_rn(d, c.T);
            const float fm = front ? 1.f : 0.f;
            const float sm_ = (!front && !back && d > 0.f) ? 1.f : 0.f;
            dsdf += gl_fs * fs_w * 2.0f * (sd * fm - fm) * fm * invRS;
            dsdf += gl_sdf * sdf_w * 2.0f * ((zz + sd * c.T) * sm_ - d * sm_) * sm_ * c.T * invRS;
            if (c.emd_w > 0.f) {
                const float gt = __fdiv_rn(__fadd_rn(__fsub_rn(d, zz), c.T), c.twoT) * 4.0f;
#pragma unroll
                for (int k = 0; k < 5; ++k)
                    dp[k] = gl_fs * c.emd_w * fm * (float)(4 - k) * invRS / 250.0f +
                            gl_sdf * c.emd_w * sm_ * fabsf(gt - (float)k) * invRS / 5000.0f;
            }
        }
        const float w = q.wt[t] * inv;
        float orgb[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) orgb[k] = G_rgb[k] * w * sg[t][k] * (1.0f - sg[t][k]);
        // rows are 40 bytes: five 8-byte stores instead of ten 4-byte ones
        float2* o2 = reinterpret_cast<float2*>(o);
        o2[0] = make_float2(orgb[0], orgb[1]); o2[1] = make_float2(orgb[2], dsdf); o2[2] = make_float2(0.f, dp[0]);
        o2[3] = make_float2(dp[1], dp[2]); o2[4] = make_float2(dp[3], dp[4]);
    }
}

// ---------------------------------------------------------------------------------------------
// Ray generation (camera -> submap frame) and its backward to the poses.
// ---------------------------------------------------------------------------------------------
// ld = floats per input record: 3 for a (R,3) direction array, 7 for the packed ray record [dir_cam | rgb | depth]
// of the keyframe ray store (mipsfusion.py:289-290,316-318), whose colour / depth columns are split out as well.
__global__ void gen_rays_kernel(const float* __restrict__ dirs, int ld, const float* __restrict__ poses,
                                const int64_t* __restrict__ pose_idx, float* __restrict__ rays_o,
                                float* __restrict__ rays_d, float* __restrict__ rgb, float* __restrict__ depth, int64_t R, int K) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= R) return;
    int64_t pi = pose_idx ? pose_idx[r] : 0;
    if (pi < 0) pi += K;                                        // python negative indexing (mipsfusion.py:313)
    const float* P = poses + pi * 16;
    const float dx = dirs[r * ld], dy = dirs[r * ld + 1], dz = dirs[r * ld + 2];
    if (rgb) { rgb[r * 3] = dirs[r * ld + 3]; rgb[r * 3 + 1] = dirs[r * ld + 4]; rgb[r * 3 + 2] = dirs[r * ld + 5]; }
    if (depth) depth[r] = dirs[r * ld + 6];
#pragma unroll
    for (int j = 0; j < 3; ++j) {
        // torch.sum(d[..., None, :] * R, -1): three products, then summed
        rays_d[r * 3 + j] = __fadd_rn(__fadd_rn(__fmul_rn(dx, P[j * 4]), __fmul_rn(dy, P[j * 4 + 1])), __fmul_rn(dz, P[j * 4 + 2]));
        rays_o[r * 3 + j] = P[j * 4 + 3];
    }
}

// d_poses (K,4,4) += backward of gen_rays: rotation block d_R[j][k] += d_d[r][j] * dir[r][k], translation d_t[j] += d_o[r][j].
// Rays of one keyframe are summed in shared memory first (up to GRB_MAX_K poses per launch; beyond that straight to global):
// one global atomic per (block, pose, entry) instead of twelve per ray.
constexpr int GRB_MAX_K = 64;
__global__ void __launch_bounds__(256) gen_rays_bwd_kernel(const float* __restrict__ dirs, int dir_stride, const int64_t* __restrict__ pose_idx,
                                                           const float* __restrict__ d_o, const float* __restrict__ d_d,
                                                           float* __restrict__ d_poses, int64_t R, int K) {
    __shared__ float acc[GRB_MAX_K * 12];
    const bool use_smem = K <= GRB_MAX_K;
    if (use_smem) {
        for (int i = threadIdx.x; i < K * 12; i += blockDim.x) acc[i] = 0.f;
        __syncthreads();
    }
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r < R) {
        int64_t pi = pose_idx ? pose_idx[r] : 0;
        if (pi < 0) pi += K;
        const float dv[3] = {dirs[r * dir_stride], dirs[r * dir_stride + 1], dirs[r * dir_stride + 2]};
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float g = d_d[r * 3 + j];
            if (use_smem) {
#pragma unroll
                for (int k = 0; k < 3; ++k) atomicAdd(&acc[pi * 12 + j * 4 + k], g * dv[k]);
                atomicAdd(&acc[pi * 12 + j * 4 + 3], d_o[r * 3 + j]);
            } else {
                float* P = d_poses + pi * 16;
#pragma unroll
                for (int k = 0; k < 3; ++k) atomicAdd(&P[j * 4 + k], g * dv[k]);
                atomicAdd(&P[j * 4 + 3], d_o[r * 3 + j]);
            }
        }
    }
    if (use_smem) {
        __syncthreads();
        for (int i = threadIdx.x; i < K * 12; i += blockDim.x) {
            const float v = acc[i];
            if (v != 0.f) atomicAdd(&d_poses[(i / 12) * 16 + (i % 12)], v);
        }
    }
}

// Deterministic mode: the same gradient without atomics.  Block k owns pose k: its threads scan the rays in a fixed strided order,
// a fixed shared-memory tree combines them, and one thread adds each entry to d_poses.  No workspace: capturable as it is.
constexpr int GRB_DET_NT = 256;
__global__ void __launch_bounds__(GRB_DET_NT) gen_rays_bwd_det_kernel(const float* __restrict__ dirs, int dir_stride,
                                                                      const int64_t* __restrict__ pose_idx, const float* __restrict__ d_o,
                                                                      const float* __restrict__ d_d, float* __restrict__ d_poses, int64_t R, int K) {
    __shared__ float red[12][GRB_DET_NT];
    const int k = blockIdx.x, t = threadIdx.x;
    float a[12];
#pragma unroll
    for (int e = 0; e < 12; ++e) a[e] = 0.f;
    for (int64_t r = t; r < R; r += GRB_DET_NT) {
        int64_t pi = pose_idx ? pose_idx[r] : 0;
        if (pi < 0) pi += K;
        if (pi != k) continue;
        const float dv[3] = {dirs[r * dir_stride], dirs[r * dir_stride + 1], dirs[r * dir_stride + 2]};
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            const float g = d_d[r * 3 + j];
#pragma unroll
            for (int c = 0; c < 3; ++c) a[j * 4 + c] = __fadd_rn(a[j * 4 + c], __fmul_rn(g, dv[c]));
            a[j * 4 + 3] = __fadd_rn(a[j * 4 + 3], d_o[r * 3 + j]);
        }
    }
#pragma unroll
    for (int e = 0; e < 12; ++e) red[e][t] = a[e];
    __syncthreads();
    for (int s = GRB_DET_NT / 2; s > 0; s >>= 1) {
        if (t < s)
#pragma unroll
            for (int e = 0; e < 12; ++e) red[e][t] = __fadd_rn(red[e][t], red[e][t + s]);
        __syncthreads();
    }
    if (t < 12) d_poses[(int64_t)k * 16 + t] = __fadd_rn(d_poses[(int64_t)k * 16 + t], red[t][0]);
}

static int gen_rays_bwd_launch(const float* dirs, int stride, const int64_t* pose_idx, const float* d_o, const float* d_d, float* d_poses,
                               int64_t R, int K, cudaStream_t st) {
    if (mf_deterministic()) gen_rays_bwd_det_kernel<<<(unsigned)K, GRB_DET_NT, 0, st>>>(dirs, stride, pose_idx, d_o, d_d, d_poses, R, K);
    else gen_rays_bwd_kernel<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(dirs, stride, pose_idx, d_o, d_d, d_poses, R, K);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
MF_API int mf_sample_z(const float* target_d, const float* u, const float* lin_uniform, const float* lin_range,
                       const float* lin_fallback, const mf_render_cfg* cfg, float* z, int64_t* counts, int64_t R, void* stream) {
    return mf_sample_z_ld(target_d, 1, u, lin_uniform, lin_range, lin_fallback, cfg, z, counts, R, stream);
}

MF_API int mf_sample_z_ld(const float* target_d, int ld_d, const float* u, const float* lin_uniform, const float* lin_range,
                          const float* lin_fallback, const mf_render_cfg* cfg, float* z, int64_t* counts, int64_t R, void* stream) {
    MF_CHECK_ARG(cfg && z && R >= 0 && ld_d >= 1);
    if (R == 0) return MF_OK;
    RenderCfgDev c = cfg_to_dev(cfg);
    c.ld_d = ld_d;
    if (!target_d) c.n_r = 0;
    const int S = c.n_u + c.n_r;
    MF_CHECK_ARG(S > 0 && S <= 4096);
    MF_CHECK_ARG(c.n_u == 0 || lin_uniform);
    MF_CHECK_ARG(c.n_r == 0 || (lin_range && lin_fallback));
    MF_CHECK_ARG(!target_d || counts);
    cudaStream_t st = (cudaStream_t)stream;
    if (counts) MF_CUDA(cudaMemsetAsync(counts, 0, 2 * sizeof(int64_t), st));
    const int threads = S <= 32 ? 32 : (S <= 64 ? 64 : 128);
    MF_CUDA(mf_launch(sample_z_kernel, (unsigned)R, threads, S * sizeof(float), st, target_d, u, lin_uniform, lin_range, lin_fallback, c, z,
                      (unsigned long long*)counts, R));
    return MF_OK;
}

MF_API int mf_render_loss_fwd(const float* raw, const float* z, const float* target_rgb, const float* target_d,
                              const int64_t* counts, const mf_render_cfg* cfg, float* out_rgb, float* out_depth,
                              float* out_aux, float* out_weights, int32_t* inds, float* losses, float* scratch, int64_t R, int S,
                              void* stream) {
    return mf_render_loss_fwd_ld(raw, z, target_rgb, 3, target_d, 1, counts, cfg, out_rgb, out_depth, out_aux, out_weights, inds, losses,
                                 scratch, R, S, stream);
}

MF_API int mf_render_loss_fwd_ld(const float* raw, const float* z, const float* target_rgb, int ld_rgb, const float* target_d, int ld_d,
                                 const int64_t* counts, const mf_render_cfg* cfg, float* out_rgb, float* out_depth,
                                 float* out_aux, float* out_weights, int32_t* inds, float* losses, float* scratch, int64_t R, int S,
                                 void* stream) {
    MF_CHECK_ARG(cfg && raw && z && out_rgb && out_depth && R >= 0 && ld_rgb >= 3 && ld_d >= 1);
    MF_CHECK_ARG(S > 0 && S <= MAX_S);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(!target_d || (counts && losses && scratch));
    RenderCfgDev c = cfg_to_dev(cfg);
    c.ld_rgb = ld_rgb; c.ld_d = ld_d;
    cudaStream_t st = (cudaStream_t)stream;
    MF_CUDA(mf_launch(render_loss_fwd_kernel, (unsigned)((R + 7) / 8), 256, 0, st, raw, z, target_rgb, target_d, c, out_rgb, out_depth, out_aux,
                      out_weights, inds, scratch, R, S));
    if (target_d) MF_CUDA(mf_launch(loss_finalize_kernel, 1, 1024, 0, st, scratch, (const unsigned long long*)counts, c, losses, R, S));
    return MF_OK;
}

static int render_loss_bwd_launch(const float* raw, const float* z, const float* target_rgb, const float* target_d,
                                  const float* losses, const mf_render_cfg* cfg, LossGrads gl, const float* g_rgb,
                                  const float* g_depth, float* d_raw, int64_t R, int S, void* stream, const char* fn, int ld_rgb = 3,
                                  int ld_d = 1) {
    if (!(cfg && raw && z && d_raw && R >= 0 && ld_rgb >= 3 && ld_d >= 1 && (((uintptr_t)d_raw & 7) == 0) && S > 0 && S <= MAX_S && (!target_d || losses))) {
        mf_set_error("%s: invalid argument", fn);
        return MF_ERR_INVALID;
    }
    if (R == 0) return MF_OK;
    RenderCfgDev c = cfg_to_dev(cfg);
    c.ld_rgb = ld_rgb; c.ld_d = ld_d;
    MF_CUDA(mf_launch(render_loss_bwd_kernel, (unsigned)((R + 7) / 8), 256, 0, (cudaStream_t)stream, raw, z, target_rgb, target_d, losses, c,
                      gl, g_rgb, g_depth, d_raw, R, S));
    return MF_OK;
}

MF_API int mf_render_loss_bwd(const float* raw, const float* z, const float* target_rgb, const float* target_d,
                              const int64_t* counts, const float* losses, const mf_render_cfg* cfg, const float* g_losses,
                              const float* g_rgb, const float* g_depth, float* d_raw, int64_t R, int S, void* stream) {
    (void)counts;
    LossGrads gl;
    for (int i = 0; i < 4; ++i) gl.p[i] = g_losses ? g_losses + i : nullptr;
    return render_loss_bwd_launch(raw, z, target_rgb, target_d, losses, cfg, gl, g_rgb, g_depth, d_raw, R, S, stream, __func__);
}

MF_API int mf_render_loss_bwd_scalars(const float* raw, const float* z, const float* target_rgb, int ld_rgb, const float* target_d, int ld_d,
                                      const float* losses, const mf_render_cfg* cfg, const float* g_rgb_loss, const float* g_depth_loss,
                                      const float* g_sdf_loss, const float* g_fs_loss, const float* g_rgb, const float* g_depth,
                                      float* d_raw, int64_t R, int S, void* stream) {
    LossGrads gl;
    gl.p[0] = g_rgb_loss; gl.p[1] = g_depth_loss; gl.p[2] = g_sdf_loss; gl.p[3] = g_fs_loss;
    return render_loss_bwd_launch(raw, z, target_rgb, target_d, losses, cfg, gl, g_rgb, g_depth, d_raw, R, S, stream, __func__, ld_rgb, ld_d);
}

MF_API int mf_gen_rays(const float* dirs_cam, const float* poses, const int64_t* pose_idx, float* rays_o, float* rays_d,
                       int64_t R, int K, void* stream) {
    MF_CHECK_ARG(R >= 0 && K >= 1);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(dirs_cam && poses && rays_o && rays_d);
    gen_rays_kernel<<<(unsigned)((R + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dirs_cam, 3, poses, pose_idx, rays_o, rays_d,
                                                                                   nullptr, nullptr, R, K);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_gen_rays_packed(const float* rays7, const float* poses, const int64_t* pose_idx, float* rays_o, float* rays_d,
                              float* target_rgb, float* target_d, int64_t R, int K, void* stream) {
    MF_CHECK_ARG(R >= 0 && K >= 1);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(rays7 && poses && rays_o && rays_d && target_rgb && target_d);
    gen_rays_kernel<<<(unsigned)((R + 255) / 256), 256, 0, (cudaStream_t)stream>>>(rays7, 7, poses, pose_idx, rays_o, rays_d,
                                                                                   target_rgb, target_d, R, K);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_gen_rays_bwd(const float* dirs_cam, const int64_t* pose_idx, const float* d_rays_o, const float* d_rays_d,
                           float* d_poses, int64_t R, int K, void* stream) {
    MF_CHECK_ARG(R >= 0 && K >= 1);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(dirs_cam && d_rays_o && d_rays_d && d_poses);
    return gen_rays_bwd_launch(dirs_cam, 3, pose_idx, d_rays_o, d_rays_d, d_poses, R, K, (cudaStream_t)stream);
}

MF_API int mf_gen_rays_packed_bwd(const float* rays7, const int64_t* pose_idx, const float* d_rays_o, const float* d_rays_d,
                                  float* d_poses, int64_t R, int K, void* stream) {
    MF_CHECK_ARG(R >= 0 && K >= 1);
    if (R == 0) return MF_OK;
    MF_CHECK_ARG(rays7 && d_rays_o && d_rays_d && d_poses);
    return gen_rays_bwd_launch(rays7, 7, pose_idx, d_rays_o, d_rays_d, d_poses, R, K, (cudaStream_t)stream);
}
