// Overlap-region SDF consistency of the inactive-map global BA (InactiveMap.py:128-192 infer_pts / get_SDF_dif /
// get_SDF_dif2, loss geometry_helper.py:225-229) for many submap pairs per call, with deterministic pose gradients.
//
// Layout: pair p uses submaps (id1, id2); the table pair_tab (P,4) int32 holds {pose1, pose2, off1, off2}: the rows of the
// two first-keyframe poses in `first_poses` and the first point row of each side's N points in the point buffer.  The host
// groups the rows by submap (all sides that query submap m are one contiguous segment), so the field is evaluated with one
// mf_field_query / mf_field_query_bwd per distinct submap.  Per-ray inputs: element (p, r) of target_d sits at
// target_d[(p N + r) ld_d], the direction at rays_d_cam[(p N + r) ld_dir + k] (row-strided views of the reference's
// (N,7) ray tensor are read in place).  ovlp: (P, N, 4, 4) (ovlp_per_ray = 1) or (P, 1, 4, 4).
// No atomics anywhere: every sum has a fixed order, so two calls give bitwise equal losses and gradients.
#include "mf_common.cuh"

// F^-1 in fp64 through the adjugate (2x2 minors of the row pairs {0,1} and {2,3}), rounded once to fp32.
__device__ __forceinline__ void inverse4_fp64(const float* __restrict__ F, float inv[16]) {
    double a[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) a[i] = (double)F[i];
    const double s0 = a[0] * a[5] - a[4] * a[1], s1 = a[0] * a[6] - a[4] * a[2], s2 = a[0] * a[7] - a[4] * a[3];
    const double s3 = a[1] * a[6] - a[5] * a[2], s4 = a[1] * a[7] - a[5] * a[3], s5 = a[2] * a[7] - a[6] * a[3];
    const double c5 = a[10] * a[15] - a[14] * a[11], c4 = a[9] * a[15] - a[13] * a[11], c3 = a[9] * a[14] - a[13] * a[10];
    const double c2 = a[8] * a[15] - a[12] * a[11], c1 = a[8] * a[14] - a[12] * a[10], c0 = a[8] * a[13] - a[12] * a[9];
    const double det = s0 * c5 - s1 * c4 + s2 * c3 + s3 * c2 - s4 * c1 + s5 * c0;
    const double b[16] = {
        a[5] * c5 - a[6] * c4 + a[7] * c3,   -a[1] * c5 + a[2] * c4 - a[3] * c3,   a[13] * s5 - a[14] * s4 + a[15] * s3,  -a[9] * s5 + a[10] * s4 - a[11] * s3,
        -a[4] * c5 + a[6] * c2 - a[7] * c1,  a[0] * c5 - a[2] * c2 + a[3] * c1,    -a[12] * s5 + a[14] * s2 - a[15] * s1, a[8] * s5 - a[10] * s2 + a[11] * s1,
        a[4] * c4 - a[5] * c2 + a[7] * c0,   -a[0] * c4 + a[1] * c2 - a[3] * c0,   a[12] * s4 - a[13] * s2 + a[15] * s0,  -a[8] * s4 + a[9] * s2 - a[11] * s0,
        -a[4] * c3 + a[5] * c1 - a[6] * c0,  a[0] * c3 - a[1] * c1 + a[2] * c0,    -a[12] * s3 + a[13] * s1 - a[14] * s0, a[8] * s3 - a[9] * s1 + a[10] * s0};
#pragma unroll
    for (int i = 0; i < 16; ++i) inv[i] = (float)(b[i] / det);
}

// A = F^-1 O (rows 0..2; row 3 of a rigid pose product is not used), fp32, k = 0..3 in order
__device__ __forceinline__ void local_pose(const float* fi, const float* __restrict__ O, float A[12]) {
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float s = __fmul_rn(fi[i * 4], O[j]);
#pragma unroll
            for (int k = 1; k < 4; ++k) s = fmaf(fi[i * 4 + k], O[k * 4 + j], s);
            A[i * 4 + j] = s;
        }
}

// infer_pts (InactiveMap.py:128-139): d = sum_k d_cam[k] A[:3,k] (products rounded, summed left to right),
// x = A[:3,3] + d * depth.  One block per (pair, side).
__global__ void __launch_bounds__(128) overlap_points_kernel(const float* __restrict__ first, const int* __restrict__ tab, int N,
                                                             const float* __restrict__ ovlp, int per_ray,
                                                             const float* __restrict__ target_d, int ld_d,
                                                             const float* __restrict__ dirs, int ld_dir,
                                                             float* __restrict__ finv, float* __restrict__ pts) {
    __shared__ float fi[16];
    const int p = blockIdx.x, s = blockIdx.y;
    if (threadIdx.x == 0) {
        float inv[16];
        inverse4_fp64(first + (size_t)tab[p * 4 + s] * 16, inv);
        for (int i = 0; i < 16; ++i) { fi[i] = inv[i]; finv[(p * 2 + s) * 16 + i] = inv[i]; }
    }
    __syncthreads();
    const int64_t off = tab[p * 4 + 2 + s];
    float A[12];
    if (!per_ray) local_pose(fi, ovlp + (size_t)p * 16, A);
    for (int r = threadIdx.x; r < N; r += blockDim.x) {
        const int64_t row = (int64_t)p * N + r;
        if (per_ray) local_pose(fi, ovlp + row * 16, A);
        const float depth = target_d[row * ld_d];
        const float dc[3] = {dirs[row * ld_dir], dirs[row * ld_dir + 1], dirs[row * ld_dir + 2]};
#pragma unroll
        for (int i = 0; i < 3; ++i) {
            const float d = __fadd_rn(__fadd_rn(__fmul_rn(dc[0], A[i * 4]), __fmul_rn(dc[1], A[i * 4 + 1])), __fmul_rn(dc[2], A[i * 4 + 2]));
            pts[(off + r) * 3 + i] = __fadd_rn(A[i * 4 + 3], __fmul_rn(d, depth));
        }
    }
}

__device__ __forceinline__ float overlap_mask(const float* target_d, int ld_d, const void* mask, int kind, int ld_m, int64_t row) {
    if (kind == 1) return reinterpret_cast<const float*>(mask)[row * ld_m];
    if (kind == 2) return reinterpret_cast<const uint8_t*>(mask)[row * ld_m] ? 1.f : 0.f;
    return target_d[row * ld_d] > 0.f ? 1.f : 0.f;               // get_SDF_dif: depth_mask = (target_d > 0)
}

constexpr int OV_NT = 256;

// compute_avg_SDF_difference (geometry_helper.py:225-229) of one pair per block: sdf = raw[:,3] * trunc,
// loss = sum (sdf1 m - sdf2 m)^2 / (count_nonzero(m) + 0.001); per-thread sums in ray order, then a fixed shared-memory tree.
// Also the d raw rows of both sides for d loss = 1 (column 3 only; rows with m = 0 exactly zero, so the field backward's
// active-point compaction skips them).  The upstream gradient of the loss is applied in overlap_pose_bwd (d_pts is linear in it).
__global__ void __launch_bounds__(OV_NT) overlap_loss_kernel(const float* __restrict__ raw, const int* __restrict__ tab, int N,
                                                             const float* __restrict__ target_d, int ld_d, const void* mask,
                                                             int mask_kind, int ld_m, float trunc, float* __restrict__ loss,
                                                             float* __restrict__ d_raw) {
    __shared__ float ssum[OV_NT];
    __shared__ int scnt[OV_NT];
    const int p = blockIdx.x, t = threadIdx.x;
    const int64_t off1 = tab[p * 4 + 2], off2 = tab[p * 4 + 3];
    float sum = 0.f; int cnt = 0;
    for (int r = t; r < N; r += OV_NT) {
        const int64_t row = (int64_t)p * N + r;
        const float m = overlap_mask(target_d, ld_d, mask, mask_kind, ld_m, row);
        const float s1 = __fmul_rn(raw[(off1 + r) * MF_RAW_DIM + 3], trunc), s2 = __fmul_rn(raw[(off2 + r) * MF_RAW_DIM + 3], trunc);
        const float a = __fsub_rn(__fmul_rn(s1, m), __fmul_rn(s2, m));
        sum = fmaf(a, a, sum);
        cnt += m != 0.f;
    }
    ssum[t] = sum; scnt[t] = cnt;
    __syncthreads();
    for (int h = OV_NT / 2; h > 0; h >>= 1) {
        if (t < h) { ssum[t] += ssum[t + h]; scnt[t] += scnt[t + h]; }
        __syncthreads();
    }
    const float denom = __fadd_rn((float)scnt[0], 0.001f);
    if (t == 0) loss[p] = __fdiv_rn(ssum[0], denom);
    const float inv = __fdiv_rn(1.f, denom);
    for (int r = t; r < N; r += OV_NT) {
        const int64_t row = (int64_t)p * N + r;
        const float m = overlap_mask(target_d, ld_d, mask, mask_kind, ld_m, row);
        float g = 0.f;
        if (m != 0.f) {
            const float s1 = __fmul_rn(raw[(off1 + r) * MF_RAW_DIM + 3], trunc), s2 = __fmul_rn(raw[(off2 + r) * MF_RAW_DIM + 3], trunc);
            const float a = __fsub_rn(__fmul_rn(s1, m), __fmul_rn(s2, m));
            g = __fmul_rn(__fmul_rn(__fmul_rn(inv, __fmul_rn(2.f, a)), m), trunc);
        }
#pragma unroll
        for (int c = 0; c < MF_RAW_DIM; ++c) {
            d_raw[(off1 + r) * MF_RAW_DIM + c] = c == 3 ? g : 0.f;
            d_raw[(off2 + r) * MF_RAW_DIM + c] = c == 3 ? -g : 0.f;
        }
    }
}

// Pose backward, one block per pair (both sides, so that d O_r = F1^-T dA1_r + F2^-T dA2_r is formed per ray in a fixed
// order without a second pass):
//   dx = g_loss[p ld_g] d_pts;  dA[:3,3] = dx;  dA[i][k] = (dx_i depth) d_cam_k;  d(F^-1) = sum_r dA_r O_r^T (per-thread sums in
//   ray order, fixed shared-memory tree);  dF = -F^-T d(F^-1) F^-T  (fp64, rounded once) -> dF_pair (P,2,16).
__global__ void __launch_bounds__(OV_NT) overlap_pose_bwd_kernel(const float* __restrict__ finv, const int* __restrict__ tab, int N,
                                                                 const float* __restrict__ ovlp, int per_ray,
                                                                 const float* __restrict__ target_d, int ld_d,
                                                                 const float* __restrict__ dirs, int ld_dir,
                                                                 const float* __restrict__ d_pts, const float* __restrict__ g_loss, int ld_g,
                                                                 float* __restrict__ dF_pair, float* __restrict__ d_ovlp) {
    __shared__ float red[24][OV_NT];
    __shared__ float fi[2][16];
    const int p = blockIdx.x, t = threadIdx.x;
    if (t < 32) fi[t >> 4][t & 15] = finv[p * 32 + t];
    __syncthreads();
    const float g = g_loss ? g_loss[(int64_t)p * ld_g] : 1.f;
    const int64_t off[2] = {tab[p * 4 + 2], tab[p * 4 + 3]};
    float acc[24];
#pragma unroll
    for (int e = 0; e < 24; ++e) acc[e] = 0.f;
    for (int r = t; r < N; r += OV_NT) {
        const int64_t row = (int64_t)p * N + r;
        const float depth = target_d[row * ld_d];
        const float dc[3] = {dirs[row * ld_dir], dirs[row * ld_dir + 1], dirs[row * ld_dir + 2]};
        const float* O = ovlp + (per_ray ? row : (int64_t)p) * 16;
        float dO[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) dO[e] = 0.f;
#pragma unroll
        for (int s = 0; s < 2; ++s) {
            float dA[12];
#pragma unroll
            for (int i = 0; i < 3; ++i) {
                const float dx = __fmul_rn(g, d_pts[(off[s] + r) * 3 + i]);
                const float dd = __fmul_rn(dx, depth);
#pragma unroll
                for (int k = 0; k < 3; ++k) dA[i * 4 + k] = __fmul_rn(dd, dc[k]);
                dA[i * 4 + 3] = dx;
            }
            if (per_ray) {
#pragma unroll
                for (int i = 0; i < 3; ++i)
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        float v = acc[s * 12 + i * 4 + j];
#pragma unroll
                        for (int l = 0; l < 4; ++l) v = fmaf(dA[i * 4 + l], O[j * 4 + l], v);
                        acc[s * 12 + i * 4 + j] = v;
                    }
                if (d_ovlp) {
#pragma unroll
                    for (int k = 0; k < 4; ++k)
#pragma unroll
                        for (int l = 0; l < 4; ++l)
#pragma unroll
                            for (int i = 0; i < 3; ++i) dO[k * 4 + l] = fmaf(fi[s][i * 4 + k], dA[i * 4 + l], dO[k * 4 + l]);
                }
            } else {
#pragma unroll
                for (int e = 0; e < 12; ++e) acc[s * 12 + e] = __fadd_rn(acc[s * 12 + e], dA[e]);
            }
        }
        if (per_ray && d_ovlp) {
#pragma unroll
            for (int e = 0; e < 16; ++e) d_ovlp[row * 16 + e] = dO[e];
        }
    }
#pragma unroll
    for (int e = 0; e < 24; ++e) red[e][t] = acc[e];
    __syncthreads();
    for (int h = OV_NT / 2; h > 0; h >>= 1) {
        if (t < h)
#pragma unroll
            for (int e = 0; e < 24; ++e) red[e][t] += red[e][t + h];
        __syncthreads();
    }
    // red[s*12 + i*4 + j][0]: d(F_s^-1)[i][j] (per-ray O) or sum_r dA[i][j] (shared O)
    if (t < 32) {
        const int s = t >> 4, a = (t >> 2) & 3, c = t & 3;
        const float* O = ovlp + (int64_t)p * 16;                     // the shared O (read only when !per_ray)
        double G[12];
#pragma unroll
        for (int i = 0; i < 3; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                double v = 0.0;
                if (per_ray) v = red[s * 12 + i * 4 + j][0];
                else
                    for (int l = 0; l < 4; ++l) v += (double)red[s * 12 + i * 4 + l][0] * O[j * 4 + l];
                G[i * 4 + j] = v;
            }
        // dF[a][c] = -sum_b (sum_i Fi[i][a] G[i][b]) Fi[c][b]
        double v = 0.0;
        for (int b = 0; b < 4; ++b) {
            double tb = 0.0;
            for (int i = 0; i < 3; ++i) tb += (double)fi[s][i * 4 + a] * G[i * 4 + b];
            v += tb * (double)fi[s][c * 4 + b];
        }
        dF_pair[(p * 2 + s) * 16 + a * 4 + c] = (float)(-v);
    }
    if (!per_ray && d_ovlp && t < 16) {                               // d O = F1^-T S1 + F2^-T S2
        const int k = t >> 2, l = t & 3;
        float v = 0.f;
        for (int s = 0; s < 2; ++s)
            for (int i = 0; i < 3; ++i) v = fmaf(fi[s][i * 4 + k], red[s * 12 + i * 4 + l][0], v);
        d_ovlp[(int64_t)p * 16 + t] = v;
    }
}

// d first_poses[m] = sum over pairs in order (side 1, then side 2) of the pair gradients of the sides that use pose m.
__global__ void overlap_first_grad_kernel(const float* __restrict__ dF_pair, const int* __restrict__ tab, int P, int n_poses,
                                          float* __restrict__ d_first) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= n_poses * 16) return;
    const int m = t >> 4, e = t & 15;
    float v = 0.f;
    for (int p = 0; p < P; ++p)
        for (int s = 0; s < 2; ++s)
            if (tab[p * 4 + s] == m) v = __fadd_rn(v, dF_pair[(p * 2 + s) * 16 + e]);
    d_first[t] = v;
}

MF_API int mf_overlap_points(const float* first_poses, const int* pair_tab, int P, int N, const float* ovlp, int ovlp_per_ray,
                             const float* target_d, int ld_d, const float* rays_d_cam, int ld_dir, float* finv, float* pts,
                             void* stream) {
    MF_CHECK_ARG(P > 0 && N > 0 && P <= 65535 && ld_d > 0 && ld_dir >= 3);
    MF_CHECK_ARG(first_poses && pair_tab && ovlp && target_d && rays_d_cam && finv && pts);
    overlap_points_kernel<<<dim3(P, 2), 128, 0, (cudaStream_t)stream>>>(first_poses, pair_tab, N, ovlp, ovlp_per_ray, target_d, ld_d,
                                                                         rays_d_cam, ld_dir, finv, pts);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_overlap_loss(const float* raw, const int* pair_tab, int P, int N, const float* target_d, int ld_d, const void* mask,
                           int mask_kind, int ld_m, double trunc, float* loss, float* d_raw, void* stream) {
    MF_CHECK_ARG(P > 0 && N > 0 && ld_d > 0 && mask_kind >= 0 && mask_kind <= 2);
    MF_CHECK_ARG(raw && pair_tab && target_d && loss && d_raw);
    MF_CHECK_ARG(mask_kind == 0 || (mask && ld_m > 0));
    overlap_loss_kernel<<<P, OV_NT, 0, (cudaStream_t)stream>>>(raw, pair_tab, N, target_d, ld_d, mask, mask_kind, ld_m, (float)trunc,
                                                              loss, d_raw);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_overlap_pose_bwd(const float* finv, const int* pair_tab, int P, int N, const float* ovlp, int ovlp_per_ray,
                               const float* target_d, int ld_d, const float* rays_d_cam, int ld_dir, const float* d_pts,
                               const float* g_loss, int ld_g, int n_poses, float* dF_pair, float* d_first, float* d_ovlp,
                               void* stream) {
    MF_CHECK_ARG(P > 0 && N > 0 && n_poses > 0 && ld_d > 0 && ld_dir >= 3 && ld_g >= 0);
    MF_CHECK_ARG(finv && pair_tab && ovlp && target_d && rays_d_cam && d_pts && dF_pair && d_first);
    cudaStream_t st = (cudaStream_t)stream;
    overlap_pose_bwd_kernel<<<P, OV_NT, 0, st>>>(finv, pair_tab, N, ovlp, ovlp_per_ray, target_d, ld_d, rays_d_cam, ld_dir, d_pts,
                                                g_loss, ld_g, dF_pair, d_ovlp);
    MF_LAUNCH_CHECK();
    overlap_first_grad_kernel<<<(n_poses * 16 + 255) / 256, 256, 0, st>>>(dF_pair, pair_tab, P, n_poses, d_first);
    MF_LAUNCH_CHECK();
    return MF_OK;
}
