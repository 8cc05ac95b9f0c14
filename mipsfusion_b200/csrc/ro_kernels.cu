// RandomOptimizer: particle pose-candidate scoring and the swarm update (a13).
// Reference: RandomOptimizer.py:54-73 (6D->7D, absolute poses), :81-85,113-131 (fitness), :202-224 (update).
#include "field_launch.cuh"
#include "field_tc_launch.cuh"

// pytorch3d.transforms.quaternion_to_matrix (real part first, two_s = 2 / |q|^2)
__device__ __forceinline__ void quat_to_mat(const float q[4], float m[9]) {
    const float r = q[0], i = q[1], j = q[2], k = q[3];
    const float two_s = 2.0f / (((r * r + i * i) + j * j) + k * k);
    m[0] = 1 - two_s * (j * j + k * k); m[1] = two_s * (i * j - k * r); m[2] = two_s * (i * k + j * r);
    m[3] = two_s * (i * j + k * r); m[4] = 1 - two_s * (i * i + k * k); m[5] = two_s * (j * k - i * r);
    m[6] = two_s * (i * k - j * r); m[7] = two_s * (j * k + i * r); m[8] = 1 - two_s * (i * i + j * j);
}

// backward of qt_to_transform_matrix (geometry_helper.py:11-17): d_c2w (rows 0-2 of a row-major 4x4) -> g[7] =
// d loss / d (quaternion, translation).  M = I + s * Q(q), s = 2 / |q|^2;  dM/dq_x = s * dQ/dq_x + Q * ds/dq_x, ds/dq_x = -s^2 q_x
__device__ __forceinline__ void qt_backward(const float q[4], const float* __restrict__ d_c2w, float g[7]) {
    const float r = q[0], i = q[1], j = q[2], k = q[3];
    const float n2 = ((r * r + i * i) + j * j) + k * k, s = 2.0f / n2;
    float G[9];
    for (int a = 0; a < 3; ++a)
        for (int b = 0; b < 3; ++b) G[a * 3 + b] = d_c2w[a * 4 + b];
    const float Q[9] = {-(j * j + k * k), i * j - k * r, i * k + j * r, i * j + k * r, -(i * i + k * k), j * k - i * r,
                        i * k - j * r, j * k + i * r, -(i * i + j * j)};
    float gq_dot = 0.f;
    for (int t = 0; t < 9; ++t) gq_dot += G[t] * Q[t];
    const float dQr[9] = {0, -k, j, k, 0, -i, -j, i, 0};
    const float dQi[9] = {0, j, k, j, -2 * i, -r, k, r, -2 * i};
    const float dQj[9] = {-2 * j, i, r, i, 0, k, -r, k, -2 * j};
    const float dQk[9] = {-2 * k, -r, i, r, -2 * k, j, i, j, 0};
    g[0] = 0.f; g[1] = 0.f; g[2] = 0.f; g[3] = 0.f; g[4] = d_c2w[3]; g[5] = d_c2w[7]; g[6] = d_c2w[11];
    for (int t = 0; t < 9; ++t) { g[0] += G[t] * dQr[t]; g[1] += G[t] * dQi[t]; g[2] += G[t] * dQj[t]; g[3] += G[t] * dQk[t]; }
    const float qv[4] = {r, i, j, k};
    for (int t = 0; t < 4; ++t) g[t] = s * g[t] - s * s * qv[t] * gq_dot;
}

// torch.optim.Adam (betas 0.9, 0.999, eps 1e-8, no weight decay) on the 7 pose parameters of a state laid out as
// [0:4] quaternion, [4:7] translation, [7:14] m, [14:21] v, [21] step count; groups: quaternion lr_rot, translation lr_trans
__device__ __forceinline__ void qt_adam_step(float* __restrict__ st, const float g[7], float lr_rot, float lr_trans) {
    const float step = st[21] + 1.f;
    st[21] = step;
    const float bc1 = 1.f - powf(0.9f, step), bc2 = 1.f - powf(0.999f, step);
    for (int t = 0; t < 7; ++t) {
        float m = st[7 + t], v = st[14 + t];
        m = 0.9f * m + 0.1f * g[t];
        v = 0.999f * v + 0.001f * g[t] * g[t];
        st[7 + t] = m; st[14 + t] = v;
        const float lr = t < 4 ? lr_rot : lr_trans;
        st[t] -= (lr / bc1) * m / (sqrtf(v) / sqrtf(bc2) + 1e-8f);
    }
}

// c2w (row-major 4x4) = qt_to_transform_matrix(q, t)
__device__ __forceinline__ void qt_to_c2w(const float q[4], const float t[3], float* __restrict__ c2w) {
    float m[9];
    quat_to_mat(q, m);
    for (int r = 0; r < 3; ++r) {
        for (int k = 0; k < 3; ++k) c2w[r * 4 + k] = m[r * 3 + k];
        c2w[r * 4 + 3] = t[r];
    }
    c2w[12] = 0.f; c2w[13] = 0.f; c2w[14] = 0.f; c2w[15] = 1.f;
}

__device__ __forceinline__ void mat3_mul(const float a[9], const float b[9], float c[9]) {
#pragma unroll
    for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int col = 0; col < 3; ++col)
            c[r * 3 + col] = fmaf(a[r * 3 + 2], b[6 + col], fmaf(a[r * 3 + 1], b[3 + col], a[r * 3] * b[col]));
}

// per candidate: rescaled particle -> 7-D pose -> absolute rotation / translation
__global__ void ro_pose_kernel(const float* __restrict__ particles6, const float* __restrict__ search_size,
                               const float* __restrict__ rot_cur, const float* __restrict__ trans_cur, int c_begin, int c_count,
                               float* __restrict__ Rt, float* __restrict__ pst7) {
    const int c = blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= c_count) return;
    float p[6];
#pragma unroll
    for (int k = 0; k < 6; ++k) p[k] = __fmul_rn(particles6[(size_t)(c_begin + c) * 6 + k], search_size[k]);
    const float imag = __fadd_rn(__fadd_rn(__fmul_rn(p[0], p[0]), __fmul_rn(p[1], p[1])), __fmul_rn(p[2], p[2]));
    const float qw = imag <= 1.0f ? sqrtf(1.0f - imag) : 0.0f;               // pose_6D_to_7D
    const float q[4] = {qw, p[0], p[1], p[2]};
    float dR[9], R0[9], R[9];
    quat_to_mat(q, dR);
#pragma unroll
    for (int k = 0; k < 9; ++k) R0[k] = rot_cur[k];
    mat3_mul(R0, dR, R);                                                      // get_abs_pose
    float* o = Rt + (size_t)c * 12;
#pragma unroll
    for (int k = 0; k < 9; ++k) o[k] = R[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) o[9 + k] = trans_cur[k] + p[3 + k];
    float* s = pst7 + (size_t)c * 7;
    s[0] = qw;
#pragma unroll
    for (int k = 0; k < 6; ++k) s[1 + k] = p[k];
}

// Point order of the scoring launch is PIXEL-major: i = pixel * C + candidate.  The 32 lanes of a warp (and the 128 points of a
// tile) are candidates of the same pixel: poses a few centimetres apart, so on the coarse and middle levels they fall into the
// same or neighbouring grid cells and their table gathers coalesce into a few cache lines instead of 32 (the gather stage of the
// forward kernel is bound by L1 wavefronts, one per distinct line).  Each point is still evaluated independently of its tile.
struct SrcRO {                             // world point of (candidate, pixel): R_c (d_cam * depth) + t_c
    const float* Rt; const float* dirs; const float* depth; int C;
    __device__ __forceinline__ void point(int64_t i, const FieldDev& f, float x[3]) const {
        const int p = (int)(i / C); const int64_t c = i % C;
        const float dp = depth[p];
        const float cam[3] = {__fmul_rn(dirs[p * 3], dp), __fmul_rn(dirs[p * 3 + 1], dp), __fmul_rn(dirs[p * 3 + 2], dp)};
        const float* R = Rt + c * 12;
        float w[3];
#pragma unroll
        for (int j = 0; j < 3; ++j)
            w[j] = __fadd_rn(fmaf(R[j * 3 + 2], cam[2], fmaf(R[j * 3 + 1], cam[1], __fmul_rn(R[j * 3], cam[0]))), R[9 + j]);
        normalize_point(f, w, x);
    }
};

struct EpiAbsSdf {                         // valid * |sdf * trunc| per (pixel, candidate)
    float* out; const float* depth; int C; float trunc;
    __device__ __forceinline__ void store(const float* OUT, int ld, int tp, int64_t tile, int64_t N, int tid, int nthreads) const {
        const int m = tid;
        const int64_t i = tile * tp + m;
        if (m < tp && i < N) {
            const float valid = depth[i / C] > 0.f ? 1.f : 0.f;
            out[i] = valid * fabsf(__fmul_rn(OUT[3 * ld + m], trunc));
        }
    }
};

// mean over the pixels of one candidate, vals[pixel][candidate].  A block owns 32 candidates: thread (cl = lane, slice = warp)
// sums the pixels slice, slice + 32, ... (coalesced over the candidates), then the 32 slice sums are added in slice order:
// a fixed summation order per candidate, independent of how the candidates are sharded.
__global__ void __launch_bounds__(1024) ro_reduce_kernel(const float* __restrict__ vals, int c_count, int P, float sdf_weight,
                                                         float* __restrict__ fitness, float* __restrict__ mean_sdf) {
    __shared__ float part[32][33];
    const int cl = threadIdx.x & 31, slice = threadIdx.x >> 5;
    const int c = blockIdx.x * 32 + cl;
    float s = 0.f;
    if (c < c_count) {
#pragma unroll 4
        for (int p = slice; p < P; p += 32) s += vals[(size_t)p * c_count + c];
    }
    part[slice][cl] = s;
    __syncthreads();
    if (slice == 0 && c < c_count) {
        float t = 0.f;
#pragma unroll
        for (int k = 0; k < 32; ++k) t += part[k][cl];
        const float mean = t / (float)P;
        mean_sdf[c] = mean;
        fitness[c] = mean * sdf_weight;
    }
}

// Swarm update (single CTA): RandomOptimizer.py:202-224
// per > 0: the three inputs are the gathered per-rank blocks [fitness (per) | mean_sdf (per) | pst7 (per x 7)] (9 per floats per
// rank, `fitness` points at the first block): candidate c lives in block c / per at row c % per -- the layout an all-gather of
// each rank's contiguous result buffer produces, read in place (no pack / unpack copies).
__device__ __forceinline__ void ro_update_body(const float* __restrict__ fitness, const float* __restrict__ mean_sdf,
                                               const float* __restrict__ pst7, int C, int per, float rescale,
                                               float* __restrict__ rot_cur, float* __restrict__ trans_cur,
                                               float* __restrict__ search_size, uint8_t* __restrict__ better_mask,
                                               int32_t* __restrict__ info) {
    __shared__ double red[32][9];
    __shared__ int red_cnt[32], red_arg[32];
    __shared__ float red_min[32];
    const float f0 = per > 0 ? __ldcg(fitness) : fitness[0];
    double acc[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};       // sum w, sum w*mean_sdf, sum w*pst7[0..6]
    int cnt = 0, arg = 0x7fffffff; float fmin_ = INFINITY;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
        const float* blk = per > 0 ? fitness + (size_t)(c / per) * 9 * per : nullptr;
        const int row = per > 0 ? c % per : c;
        const float* msdf_ = per > 0 ? blk + per : mean_sdf;
        const float* p7_ = per > 0 ? blk + 2 * per : pst7;
        const float f = per > 0 ? __ldcg(blk + row) : fitness[c];
        const bool better = f < f0;
        if (better_mask) better_mask[c] = better ? 1 : 0;
        if (f < fmin_) { fmin_ = f; arg = c; }
        if (better) {
            const float w = f0 - f;
            cnt += 1;
            acc[0] += (double)w;
            acc[1] += (double)(w * (per > 0 ? __ldcg(msdf_ + row) : msdf_[row]));
#pragma unroll
            for (int k = 0; k < 7; ++k) acc[2 + k] += (double)((per > 0 ? __ldcg(p7_ + (size_t)row * 7 + k) : p7_[(size_t)row * 7 + k]) * w);
        }
    }
    const int w_ = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int k = 0; k < 9; ++k) acc[k] = warp_sum_d(acc[k]);
    for (int o = 16; o > 0; o >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
        const float of = __shfl_xor_sync(0xffffffffu, fmin_, o);
        const int oa = __shfl_xor_sync(0xffffffffu, arg, o);
        if (of < fmin_ || (of == fmin_ && oa < arg)) { fmin_ = of; arg = oa; }
    }
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < 9; ++k) red[w_][k] = acc[k];
        red_cnt[w_] = cnt; red_arg[w_] = arg; red_min[w_] = fmin_;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double t[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    int count = 0, amin = 0x7fffffff; float vmin = INFINITY;
    const int nw = blockDim.x >> 5;
    for (int i = 0; i < nw; ++i) {
        for (int k = 0; k < 9; ++k) t[k] += red[i][k];
        count += red_cnt[i];
        if (red_min[i] < vmin || (red_min[i] == vmin && red_arg[i] < amin)) { vmin = red_min[i]; amin = red_arg[i]; }
    }
    const bool success = count > 0;
    const float wsum = (float)t[0] + 0.00001f;
    float mean_s, mt6[6];
    if (success) {
        mean_s = (float)t[1] / wsum;
        float mt[7];
        for (int k = 0; k < 7; ++k) mt[k] = (float)t[2 + k] / wsum;
        const float nrm = sqrtf(((mt[0] * mt[0] + mt[1] * mt[1]) + mt[2] * mt[2]) + mt[3] * mt[3]) + 1e-5f;
        float q[4];
        for (int k = 0; k < 4; ++k) q[k] = mt[k] / nrm;
        float dR[9], R0[9], R[9];
        quat_to_mat(q, dR);
        for (int k = 0; k < 9; ++k) R0[k] = rot_cur[k];
        mat3_mul(R0, dR, R);                                           // update_cur_pose
        for (int k = 0; k < 9; ++k) rot_cur[k] = R[k];
        for (int k = 0; k < 3; ++k) trans_cur[k] += mt[4 + k];
        mt6[0] = q[1]; mt6[1] = q[2]; mt6[2] = q[3]; mt6[3] = mt[4]; mt6[4] = mt[5]; mt6[5] = mt[6];
    } else {
        mean_s = per > 0 ? __ldcg(fitness + per) : mean_sdf[0];
        for (int k = 0; k < 6; ++k) mt6[k] = 0.f;                      // no_rel_trans[1:]
    }
    float s[6], n2 = 0.f;
    for (int k = 0; k < 6; ++k) { s[k] = fabsf(mt6[k]) + 0.0001f; n2 += s[k] * s[k]; }
    const float nrm = sqrtf(n2);
    for (int k = 0; k < 6; ++k) {
        const float ss = rescale * mean_s * s[k] / nrm + 0.0001f;      // update_search_size
        search_size[k] = success ? ss : ss * 2.0f;
    }
    if (info) { info[0] = count; info[1] = success ? 1 : 0; info[2] = amin; info[3] = 0; }
}

__global__ void __launch_bounds__(1024) ro_update_kernel(const float* __restrict__ fitness, const float* __restrict__ mean_sdf,
                                                         const float* __restrict__ pst7, int C, int per, float rescale,
                                                         float* __restrict__ rot_cur, float* __restrict__ trans_cur,
                                                         float* __restrict__ search_size, uint8_t* __restrict__ better_mask,
                                                         int32_t* __restrict__ info) {
    ro_update_body(fitness, mean_sdf, pst7, C, per, rescale, rot_cur, trans_cur, search_size, better_mask, info);
}

// Multi-GPU iteration without a collective library call: every rank's update kernel first stores its own result block
// (9 per floats) into the gathered buffer of EVERY rank over NVLink peer memory, publishes a sequence number in every rank's
// flag array (release, system scope), waits until all ranks' numbers have arrived in its own flag array (acquire), and then
// runs the swarm update on its local copy of the gathered blocks -- exchange and update are one single-CTA kernel.
// The gathered buffer is double-buffered by the parity of the sequence number: a rank can publish iteration i + 1 only after
// its own update of iteration i, and nobody can start i + 2 before everybody published i + 1 (DESIGN.md 5).
constexpr int RO_MAX_PEERS = 16;
struct RoPeers { float* gathered[RO_MAX_PEERS]; unsigned int* flags[RO_MAX_PEERS]; };

__global__ void __launch_bounds__(1024) ro_update_peer_kernel(const float* __restrict__ local_block, RoPeers peers, int rank, int world,
                                                              unsigned int seq, int C, int per, float rescale,
                                                              float* __restrict__ rot_cur, float* __restrict__ trans_cur,
                                                              float* __restrict__ search_size, uint8_t* __restrict__ better_mask,
                                                              int32_t* __restrict__ info, int* __restrict__ err) {
    const int n = 9 * per;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const float v = local_block[i];
        for (int r = 0; r < world; ++r) __stcg(peers.gathered[r] + (size_t)rank * n + i, v);
    }
    __threadfence_system();
    __syncthreads();
    if ((int)threadIdx.x < world) {
        const int r = threadIdx.x;
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(peers.flags[r] + rank), "r"(seq) : "memory");
        // wait for rank r's block (bounded: a missing peer must not hang the GPU)
        const unsigned int* mine = peers.flags[rank] + r;
        unsigned int got = 0;
        for (long long it = 0; it < (1ll << 28); ++it) {
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(got) : "l"(mine) : "memory");
            if ((int)(got - seq) >= 0) break;
        }
        if ((int)(got - seq) < 0 && err) atomicExch(err, 1);
    }
    __syncthreads();
    ro_update_body(peers.gathered[rank], nullptr, nullptr, C, per, rescale, rot_cur, trans_cur, search_size, better_mask, info);
}

MF_API int mf_ro_score(const float* particles6, const float* search_size, const float* rot_cur, const float* trans_cur,
                       const float* dirs_cam, const float* target_d, const mf_field* field, double trunc, double sdf_weight,
                       int c_begin, int c_count, int P, float* fitness, float* mean_sdf, float* pst7, float* scratch, void* stream) {
    MF_CHECK_ARG(c_begin >= 0 && c_count >= 0 && P > 0);
    if (c_count == 0) return MF_OK;
    MF_CHECK_ARG(particles6 && search_size && rot_cur && trans_cur && dirs_cam && target_d && fitness && mean_sdf && pst7 && scratch);
    FieldDev d; int rc = mf_field_to_dev(field, &d); if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    float* Rt = scratch;                                   // c_count * 12
    float* vals = scratch + (size_t)c_count * 12;          // P * c_count, pixel-major
    ro_pose_kernel<<<(c_count + 127) / 128, 128, 0, st>>>(particles6, search_size, rot_cur, trans_cur, c_begin, c_count, Rt, pst7);
    MF_LAUNCH_CHECK();
    SrcRO src{Rt, dirs_cam, target_d, c_count};
    EpiAbsSdf epi{vals, target_d, c_count, (float)trunc};
    rc = launch_field_fwd_auto<SrcRO, EpiAbsSdf, true>(d, src, epi, (int64_t)c_count * P, st, nullptr, false, 2);
    if (rc) return rc;
    ro_reduce_kernel<<<(c_count + 31) / 32, 1024, 0, st>>>(vals, c_count, P, (float)sdf_weight, fitness, mean_sdf);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_ro_update(const float* fitness, const float* mean_sdf, const float* pst7, int C, double rescale, float* rot_cur,
                        float* trans_cur, float* search_size, uint8_t* better_mask, int32_t* info, void* stream) {
    MF_CHECK_ARG(C > 0 && fitness && mean_sdf && pst7 && rot_cur && trans_cur && search_size);
    ro_update_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(fitness, mean_sdf, pst7, C, 0, (float)rescale, rot_cur, trans_cur,
                                                           search_size, better_mask, info);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_ro_update_peer(const float* local_block, const uint64_t* peer_bases, int world, int rank, int64_t off_gathered,
                             int64_t off_flags, unsigned int seq, int C, int per, double rescale, float* rot_cur, float* trans_cur,
                             float* search_size, uint8_t* better_mask, int32_t* info, void* stream) {
    MF_CHECK_ARG(local_block && peer_bases && world >= 1 && world <= RO_MAX_PEERS && rank >= 0 && rank < world);
    MF_CHECK_ARG(C > 0 && per > 0 && (int64_t)per * world >= C && rot_cur && trans_cur && search_size && off_gathered >= 0 && off_flags >= 0);
    RoPeers peers;
    const int64_t n = 9 * (int64_t)per * world;
    for (int r = 0; r < world; ++r) {
        MF_CHECK_ARG(peer_bases[r]);
        float* base = reinterpret_cast<float*>(peer_bases[r]);
        peers.gathered[r] = base + off_gathered + (seq & 1u) * n;           // double-buffered by the parity of the sequence number
        peers.flags[r] = reinterpret_cast<unsigned int*>(base + off_flags);
    }
    ro_update_peer_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(local_block, peers, rank, world, seq, C, per, (float)rescale, rot_cur,
                                                                trans_cur, search_size, better_mask, info, mf_tc_error_flag());
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_ro_update_gathered(const float* gathered, int C, int per, double rescale, float* rot_cur, float* trans_cur,
                                 float* search_size, uint8_t* better_mask, int32_t* info, void* stream) {
    MF_CHECK_ARG(C > 0 && per > 0 && gathered && rot_cur && trans_cur && search_size);
    ro_update_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(gathered, nullptr, nullptr, C, per, (float)rescale, rot_cur, trans_cur,
                                                           search_size, better_mask, info);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Gradient pose refinement of tracking (mipsfusion.py:501-556): pose parameters, their gradient and Adam on the device.
// ---------------------------------------------------------------------------------------------
__global__ void pose_to_c2w_kernel(const float* __restrict__ state, float* __restrict__ c2w) {
    if (threadIdx.x != 0) return;
    qt_to_c2w(state, state + 4, c2w);                                    // qt_to_transform_matrix, geometry_helper.py:11-17
}

__global__ void pose_refine_update_kernel(float* __restrict__ st, const float* __restrict__ c2w, const float* __restrict__ d_c2w,
                                          const float* __restrict__ losses, const float* __restrict__ loss_w, float lr_rot,
                                          float lr_trans, int wait_iters, float* __restrict__ best_c2w) {
    if (threadIdx.x != 0) return;
    if (st[24] != 0.f) return;                                           // the reference has left the loop (:551-552)
    // get_loss_from_ret (mipsfusion.py:141-152): weighted sum in the reference's order rgb, depth, sdf, fs
    float loss = 0.f;
    loss += loss_w[0] * losses[0];
    loss += loss_w[1] * losses[1];
    loss += loss_w[2] * losses[2];
    loss += loss_w[3] * losses[3];
    if (st[22] < 0.f) {                                                  // first iteration: best = this pose (:540-542)
        st[22] = loss;
        for (int k = 0; k < 16; ++k) best_c2w[k] = c2w[k];
    }
    if (loss < st[22]) {                                                 // (:546-550)
        st[22] = loss;
        for (int k = 0; k < 16; ++k) best_c2w[k] = c2w[k];
        st[23] = 0.f;
    } else {
        st[23] += 1.f;
    }
    if (st[23] > (float)wait_iters) { st[24] = 1.f; return; }            // break before backward / step
    // ---- backward of qt_to_transform_matrix, then one torch.optim.Adam step with the groups quaternion / translation ----
    const float q[4] = {st[0], st[1], st[2], st[3]};
    float g[7];
    qt_backward(q, d_c2w, g);
    qt_adam_step(st, g, lr_rot, lr_trans);
}

MF_API int mf_pose_to_c2w(const float* state, float* c2w, void* stream) {
    MF_CHECK_ARG(state && c2w);
    pose_to_c2w_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(state, c2w);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_pose_refine_update(float* state, const float* c2w, const float* d_c2w, const float* losses, const float* loss_w,
                                 double lr_rot, double lr_trans, int wait_iters, float* best_c2w, void* stream) {
    MF_CHECK_ARG(state && c2w && d_c2w && losses && loss_w && best_c2w);
    pose_refine_update_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(state, c2w, d_c2w, losses, loss_w, (float)lr_rot, (float)lr_trans,
                                                                 wait_iters, best_c2w);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Keyframe pose optimisation of the mapping loop (local_BA, mipsfusion.py:259-370; get_pose_param_optim :235-241,280-282;
// pose step :338-342): K pose states of BA_STATE floats, one thread per pose.
// ---------------------------------------------------------------------------------------------
constexpr int BA_STATE = 24;

// pytorch3d matrix_to_quaternion (rotation_conversions.py) for one row-major 3x3 block of a 4x4, in the op order of the
// torch formula (tracker.matrix_to_quaternion): real part first, standardised to a non-negative real part
__device__ __forceinline__ void mat_to_quat(const float* __restrict__ P, float q[4]) {
    const float m00 = P[0], m01 = P[1], m02 = P[2], m10 = P[4], m11 = P[5], m12 = P[6], m20 = P[8], m21 = P[9], m22 = P[10];
    const float qa[4] = {__fadd_rn(__fadd_rn(__fadd_rn(1.0f, m00), m11), m22), __fsub_rn(__fsub_rn(__fadd_rn(1.0f, m00), m11), m22),
                         __fsub_rn(__fadd_rn(__fsub_rn(1.0f, m00), m11), m22), __fadd_rn(__fsub_rn(__fsub_rn(1.0f, m00), m11), m22)};
    float q_abs[4];
    for (int a = 0; a < 4; ++a) q_abs[a] = qa[a] > 0.f ? __fsqrt_rn(qa[a]) : 0.f;
    int best = 0;                                                        // torch.argmax: the first of equal maxima
    for (int a = 1; a < 4; ++a)
        if (q_abs[a] > q_abs[best]) best = a;
    float c[4];
    const float sq = __fmul_rn(q_abs[best], q_abs[best]);
    switch (best) {
        case 0: c[0] = sq; c[1] = __fsub_rn(m21, m12); c[2] = __fsub_rn(m02, m20); c[3] = __fsub_rn(m10, m01); break;
        case 1: c[0] = __fsub_rn(m21, m12); c[1] = sq; c[2] = __fadd_rn(m10, m01); c[3] = __fadd_rn(m02, m20); break;
        case 2: c[0] = __fsub_rn(m02, m20); c[1] = __fadd_rn(m10, m01); c[2] = sq; c[3] = __fadd_rn(m12, m21); break;
        default: c[0] = __fsub_rn(m10, m01); c[1] = __fadd_rn(m20, m02); c[2] = __fadd_rn(m21, m12); c[3] = sq; break;
    }
    const float den = __fmul_rn(2.0f, fmaxf(q_abs[best], 0.1f));
    for (int a = 0; a < 4; ++a) q[a] = __fdiv_rn(c[a], den);
    if (q[0] < 0.f)
        for (int a = 0; a < 4; ++a) q[a] = -q[a];
}

__global__ void ba_pose_init_kernel(const float* __restrict__ poses, const uint8_t* __restrict__ frozen, int K,
                                    float* __restrict__ state, float* __restrict__ poses_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    const float* P = poses + k * 16;
    float* s = state + k * BA_STATE;
    for (int t = 0; t < BA_STATE; ++t) s[t] = 0.f;
    if (frozen && frozen[k]) {                                           // not a parameter: copied through bit for bit
        for (int t = 0; t < 16; ++t) poses_out[k * 16 + t] = P[t];
        return;
    }
    float q[4];
    mat_to_quat(P, q);
    for (int t = 0; t < 4; ++t) s[t] = q[t];
    s[4] = P[3]; s[5] = P[7]; s[6] = P[11];
    qt_to_c2w(s, s + 4, poses_out + k * 16);                             // poses_all is built from the parameters (:280-282)
}

__global__ void ba_pose_update_kernel(float* __restrict__ state, float* __restrict__ d_poses, const uint8_t* __restrict__ frozen,
                                      int K, float lr_rot, float lr_trans, float* __restrict__ poses_out) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    float* dP = d_poses + k * 16;
    if (!(frozen && frozen[k])) {
        float* s = state + k * BA_STATE;
        const float q[4] = {s[0], s[1], s[2], s[3]};
        float g[7];
        qt_backward(q, dP, g);
        qt_adam_step(s, g, lr_rot, lr_trans);
        qt_to_c2w(s, s + 4, poses_out + k * 16);
    }
    for (int t = 0; t < 16; ++t) dP[t] = 0.f;                            // pose_optimizer.zero_grad() after the step (:338-342)
}

// RO -> GO hand-off of tracking (mipsfusion.py:483-485,501-503): the RandomOptimizer's pose becomes c2w
// (pose_compose, geometry_helper.py:43-47) and the GO stage's parameters (matrix_to_quaternion + translation, fresh Adam state,
// no best loss yet), the state FusedPoseRefiner.refine builds on the host
__global__ void track_handoff_kernel(const float* __restrict__ rot_cur, const float* __restrict__ trans_cur,
                                     float* __restrict__ c2w, float* __restrict__ st) {
    const int t = threadIdx.x;
    if (t < 16) {
        const int r = t >> 2, c = t & 3;
        c2w[t] = r == 3 ? (c == 3 ? 1.f : 0.f) : (c == 3 ? trans_cur[r] : rot_cur[r * 3 + c]);
    }
    if (t != 0) return;
    const float P[12] = {rot_cur[0], rot_cur[1], rot_cur[2], trans_cur[0], rot_cur[3], rot_cur[4], rot_cur[5], trans_cur[1],
                         rot_cur[6], rot_cur[7], rot_cur[8], trans_cur[2]};
    float q[4];
    mat_to_quat(P, q);
    for (int k = 0; k < 32; ++k) st[k] = 0.f;
    for (int k = 0; k < 4; ++k) st[k] = q[k];
    for (int k = 0; k < 3; ++k) st[4 + k] = P[k * 4 + 3];
    st[22] = -1.f;
}

MF_API int mf_track_handoff(const float* rot_cur, const float* trans_cur, float* c2w_out, float* go_state, void* stream) {
    MF_CHECK_ARG(rot_cur && trans_cur && c2w_out && go_state);
    track_handoff_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(rot_cur, trans_cur, c2w_out, go_state);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_ba_pose_init(const float* poses, const uint8_t* frozen, int K, float* state, float* poses_out, void* stream) {
    MF_CHECK_ARG(poses && state && poses_out && K > 0);
    ba_pose_init_kernel<<<(K + 63) / 64, 64, 0, (cudaStream_t)stream>>>(poses, frozen, K, state, poses_out);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_ba_pose_update(float* state, float* d_poses, const uint8_t* frozen, int K, double lr_rot, double lr_trans,
                             float* poses_out, void* stream) {
    MF_CHECK_ARG(state && d_poses && poses_out && K > 0);
    ba_pose_update_kernel<<<(K + 63) / 64, 64, 0, (cudaStream_t)stream>>>(state, d_poses, frozen, K, (float)lr_rot, (float)lr_trans,
                                                                       poses_out);
    MF_LAUNCH_CHECK();
    return MF_OK;
}
