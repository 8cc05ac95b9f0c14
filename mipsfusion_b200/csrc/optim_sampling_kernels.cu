// Dense Adam (a10) and the integer-exact pixel samplers (a11).
// Reference: mipsfusion.py:580-584 (torch.optim.Adam configuration), torch's single-tensor Adam op order;
// helper_functions/sampling_helper.py:7-68.
#include "mf_common.cuh"

// ---------------------------------------------------------------------------------------------
// Adam.  One pass over (p, g, m, v): 16 B read + 12 B write (+4 B when the gradient is cleared)
// per parameter -- a pure HBM stream.
// ---------------------------------------------------------------------------------------------
struct AdamScalars {
    float w1;          // fp32(1 - beta1): lerp weight
    float beta2, w2;   // fp32(beta2), fp32(1 - beta2)
    float neg_step;    // fp32(-lr / (1 - beta1^t))
    float bc2_sqrt;    // fp32(sqrt(1 - beta2^t))
    float eps, wd;
};

__device__ __forceinline__ void adam_one(float& p, float& g, float& m, float& v, const AdamScalars& a) {
    float gg = g;
    if (a.wd != 0.f) gg = fmaf(a.wd, p, gg);                        // grad.add(param, alpha=wd)
    m = fmaf(gg - m, a.w1, m);                                      // exp_avg.lerp_(grad, 1 - beta1)
    v = fmaf(a.w2 * gg, gg, v * a.beta2);                           // mul_(beta2).addcmul_(g, g, 1 - beta2)
    const float denom = __fadd_rn(__fdiv_rn(sqrtf(v), a.bc2_sqrt), a.eps);
    p = fmaf(a.neg_step, __fdiv_rn(m, denom), p);                   // addcdiv_(m, denom, value=-step_size)
}

template <bool ZERO>
__global__ void __launch_bounds__(256) adam_kernel_v4(float4* __restrict__ p, float4* __restrict__ g, float4* __restrict__ m,
                                                      float4* __restrict__ v, int64_t n4, AdamScalars a) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 pp = p[i], gg = g[i], mm = m[i], vv = v[i];
        adam_one(pp.x, gg.x, mm.x, vv.x, a); adam_one(pp.y, gg.y, mm.y, vv.y, a);
        adam_one(pp.z, gg.z, mm.z, vv.z, a); adam_one(pp.w, gg.w, mm.w, vv.w, a);
        p[i] = pp; m[i] = mm; v[i] = vv;
        if (ZERO) g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

template <bool ZERO>
__global__ void adam_kernel_scalar(float* __restrict__ p, float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                   int64_t begin, int64_t n, AdamScalars a) {
    const int64_t i = begin + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float pp = p[i], gg = g[i], mm = m[i], vv = v[i];
    adam_one(pp, gg, mm, vv, a);
    p[i] = pp; m[i] = mm; v[i] = vv;
    if (ZERO) g[i] = 0.f;
}

MF_API int mf_adam_step(float* p, float* g, float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps,
                        double weight_decay, int step, int zero_grad, void* stream) {
    MF_CHECK_ARG(n >= 0 && step >= 1);
    if (n == 0) return MF_OK;
    MF_CHECK_ARG(p && g && m && v);
    AdamScalars a;
    a.w1 = (float)(1.0 - beta1); a.beta2 = (float)beta2; a.w2 = (float)(1.0 - beta2);
    a.neg_step = (float)(-(lr / (1.0 - pow(beta1, (double)step))));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(beta2, (double)step));
    a.eps = (float)eps; a.wd = (float)weight_decay;
    cudaStream_t st = (cudaStream_t)stream;
    const bool aligned = (((uintptr_t)p | (uintptr_t)g | (uintptr_t)m | (uintptr_t)v) & 15) == 0;
    const int64_t n4 = aligned ? n / 4 : 0;
    if (n4 > 0) {
        const int64_t want = (n4 + 255) / 256;
        const int64_t cap = (int64_t)mf_sm_count_cached() * 8;
        const unsigned blocks = (unsigned)(want < cap ? want : cap);
        if (zero_grad) adam_kernel_v4<true><<<blocks, 256, 0, st>>>((float4*)p, (float4*)g, (float4*)m, (float4*)v, n4, a);
        else adam_kernel_v4<false><<<blocks, 256, 0, st>>>((float4*)p, (float4*)g, (float4*)m, (float4*)v, n4, a);
        MF_LAUNCH_CHECK();
    }
    const int64_t rest = n - n4 * 4;
    if (rest > 0) {
        const unsigned blocks = (unsigned)((rest + 255) / 256);
        if (zero_grad) adam_kernel_scalar<true><<<blocks, 256, 0, st>>>(p, g, m, v, n4 * 4, n, a);
        else adam_kernel_scalar<false><<<blocks, 256, 0, st>>>(p, g, m, v, n4 * 4, n, a);
        MF_LAUNCH_CHECK();
    }
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Data-parallel mapping: gradient reduce-scatter + Adam + parameter all-gather in ONE kernel over NVLink peer memory.
// Every rank holds the same arena layout in symmetric (peer-mapped) memory; rank r owns the r-th slab of the
// parameters: it reads that slab of the gradient from every rank (fixed rank order -> all replicas receive bit-identical
// parameters), averages, applies Adam with its slab of the moments and stores the new parameters into every rank's
// copy.  Per GPU the links carry 2 (W-1)/W of the parameter bytes instead of a full all-reduce followed by a replicated
// Adam pass, and the moments are only touched on the owning rank.  The caller brackets the launch with cross-GPU barriers.
// ---------------------------------------------------------------------------------------------
constexpr int MF_MAX_PEERS = 16;
struct PeerPtrs { float* p[MF_MAX_PEERS]; const float* g[MF_MAX_PEERS]; };

// W > 0: compile-time world size (all peer loads of an element are in flight together: the slab is small, so the kernel
// is bound by NVLink latency unless every thread keeps W loads outstanding); W == 0: run-time world size.
// MC: the arena also has an NVSwitch multicast mapping (NVLS): the gradient sum over all ranks is one
// multimem.ld_reduce (reduced inside the switch) and the new parameters reach all replicas with one multimem.st, which
// roughly halves the bytes each GPU's links carry.
__device__ __forceinline__ float4 multimem_ld_reduce_add(const float4* mc) {
    float4 r;
    asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                 : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(mc) : "memory");
    return r;
}
__device__ __forceinline__ void multimem_st(float4* mc, float4 v) {
    asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(mc), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}

template <int W, bool MC>
__global__ void __launch_bounds__(256) adam_sharded_kernel(PeerPtrs peers, int world_rt, float inv_world, float4* __restrict__ m,
                                                           float4* __restrict__ v, float4* __restrict__ g_clear, int64_t begin4,
                                                           int64_t end4, int64_t n4, AdamScalars a, const float4* mc_g, float4* mc_p) {
    const int world = W > 0 ? W : world_rt;
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, t0 = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    for (int64_t i = begin4 + t0; i < end4; i += stride) {
        float4 gg;
        if (MC) {
            gg = multimem_ld_reduce_add(mc_g + i);
        } else if (W > 0) {
            float4 gs[W > 0 ? W : 1];
#pragma unroll
            for (int r = 0; r < W; ++r) gs[r] = reinterpret_cast<const float4*>(peers.g[r])[i];
            gg = gs[0];
#pragma unroll
            for (int r = 1; r < W; ++r) { gg.x += gs[r].x; gg.y += gs[r].y; gg.z += gs[r].z; gg.w += gs[r].w; }
        } else {
            gg = reinterpret_cast<const float4*>(peers.g[0])[i];
            for (int r = 1; r < world; ++r) {
                const float4 o = reinterpret_cast<const float4*>(peers.g[r])[i];
                gg.x += o.x; gg.y += o.y; gg.z += o.z; gg.w += o.w;
            }
        }
        gg.x *= inv_world; gg.y *= inv_world; gg.z *= inv_world; gg.w *= inv_world;
        float4 pp = reinterpret_cast<const float4*>(peers.p[0])[i];      // slot 0 = the local copy; all replicas are identical
        float4 mm = m[i], vv = v[i];
        adam_one(pp.x, gg.x, mm.x, vv.x, a); adam_one(pp.y, gg.y, mm.y, vv.y, a);
        adam_one(pp.z, gg.z, mm.z, vv.z, a); adam_one(pp.w, gg.w, mm.w, vv.w, a);
        m[i] = mm; v[i] = vv;
        if (MC) {
            multimem_st(mc_p + i, pp);
        } else {
#pragma unroll
            for (int r = 0; r < (W > 0 ? W : world); ++r) reinterpret_cast<float4*>(peers.p[r])[i] = pp;
        }
    }
    if (g_clear)                                                         // zero_grad of the buffer the NEXT backward accumulates into
        for (int64_t i = t0; i < n4; i += stride) g_clear[i] = make_float4(0.f, 0.f, 0.f, 0.f);
}

MF_API int mf_adam_step_sharded(const uint64_t* peer_bases, int world, int rank, int64_t off_p, int64_t off_g, int64_t off_g_clear,
                                float* m, float* v, int64_t n, double lr, double beta1, double beta2, double eps,
                                double weight_decay, int step, uint64_t multicast_base, void* stream) {
    MF_CHECK_ARG(peer_bases && world >= 1 && world <= MF_MAX_PEERS && rank >= 0 && rank < world);
    MF_CHECK_ARG(n >= 0 && (n & 3) == 0 && step >= 1 && m && v);
    MF_CHECK_ARG(((off_p | off_g) & 3) == 0 && (off_g_clear < 0 || (off_g_clear & 3) == 0));
    if (n == 0) return MF_OK;
    PeerPtrs peers;
    for (int r = 0; r < world; ++r) {
        MF_CHECK_ARG(peer_bases[r] && (peer_bases[r] & 15) == 0);
        peers.p[r] = reinterpret_cast<float*>(peer_bases[r]) + off_p;
        peers.g[r] = reinterpret_cast<const float*>(peer_bases[r]) + off_g;
    }
    // the kernel reads the parameters through slot 0 and writes through every slot: put the local copy in slot 0
    { float* t = peers.p[0]; peers.p[0] = peers.p[rank]; peers.p[rank] = t; }
    MF_CHECK_ARG((((uintptr_t)m | (uintptr_t)v) & 15) == 0);
    AdamScalars a;
    a.w1 = (float)(1.0 - beta1); a.beta2 = (float)beta2; a.w2 = (float)(1.0 - beta2);
    a.neg_step = (float)(-(lr / (1.0 - pow(beta1, (double)step))));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(beta2, (double)step));
    a.eps = (float)eps; a.wd = (float)weight_decay;
    const int64_t n4 = n / 4, per = (n4 + world - 1) / world;
    const int64_t begin4 = per * rank < n4 ? per * rank : n4, end4 = begin4 + per < n4 ? begin4 + per : n4;
    float4* clear = off_g_clear >= 0 ? reinterpret_cast<float4*>(reinterpret_cast<float*>(peer_bases[rank]) + off_g_clear) : nullptr;
    const int64_t work = clear ? n4 : (end4 - begin4);
    const int64_t want = (work + 255) / 256, cap = (int64_t)mf_sm_count_cached() * 8;
    const unsigned blocks = (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
    cudaStream_t st = (cudaStream_t)stream;
    const float inv = (float)(1.0 / world);
    MF_CHECK_ARG((multicast_base & 15) == 0);
    const float4* mc_g = multicast_base ? reinterpret_cast<const float4*>(reinterpret_cast<const float*>(multicast_base) + off_g) : nullptr;
    float4* mc_p = multicast_base ? reinterpret_cast<float4*>(reinterpret_cast<float*>(multicast_base) + off_p) : nullptr;
#define MF_LAUNCH_SHARDED(W, MC) adam_sharded_kernel<W, MC><<<blocks, 256, 0, st>>>(peers, world, inv, (float4*)m, (float4*)v, clear, \
                                                                                    begin4, end4, n4, a, mc_g, mc_p)
    if (multicast_base) {
        MF_LAUNCH_SHARDED(0, true);
    } else {
        switch (world) {
            case 2: MF_LAUNCH_SHARDED(2, false); break;
            case 4: MF_LAUNCH_SHARDED(4, false); break;
            case 8: MF_LAUNCH_SHARDED(8, false); break;
            default: MF_LAUNCH_SHARDED(0, false); break;
        }
    }
#undef MF_LAUNCH_SHARDED
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// Two tensors with their own hyper-parameters in ONE launch (the hash grid and the decoder blob of a mapping step): the
// first b0 blocks stride over tensor 0, the remaining blocks over tensor 1.  Both lengths must be multiples of 4.
struct AdamTensor { float4 *p, *g, *m, *v; int64_t n4; AdamScalars a; };

__global__ void __launch_bounds__(256) adam_pair_kernel(AdamTensor t0, AdamTensor t1, int b0) {
    const bool first = (int)blockIdx.x < b0;
    const AdamTensor& t = first ? t0 : t1;
    const int64_t nb = first ? b0 : (int)gridDim.x - b0, bi = first ? blockIdx.x : blockIdx.x - b0;
    for (int64_t i = bi * blockDim.x + threadIdx.x; i < t.n4; i += nb * blockDim.x) {
        float4 pp = t.p[i], gg = t.g[i], mm = t.m[i], vv = t.v[i];
        adam_one(pp.x, gg.x, mm.x, vv.x, t.a); adam_one(pp.y, gg.y, mm.y, vv.y, t.a);
        adam_one(pp.z, gg.z, mm.z, vv.z, t.a); adam_one(pp.w, gg.w, mm.w, vv.w, t.a);
        t.p[i] = pp; t.m[i] = mm; t.v[i] = vv;
        t.g[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

static AdamScalars adam_scalars(double lr, double beta1, double beta2, double eps, double weight_decay, int step) {
    AdamScalars a;
    a.w1 = (float)(1.0 - beta1); a.beta2 = (float)beta2; a.w2 = (float)(1.0 - beta2);
    a.neg_step = (float)(-(lr / (1.0 - pow(beta1, (double)step))));
    a.bc2_sqrt = (float)sqrt(1.0 - pow(beta2, (double)step));
    a.eps = (float)eps; a.wd = (float)weight_decay;
    return a;
}

MF_API int mf_adam_step_pair(float* p0, float* g0, float* m0, float* v0, int64_t n0, double lr0, double eps0, double wd0,
                             float* p1, float* g1, float* m1, float* v1, int64_t n1, double lr1, double eps1, double wd1,
                             double beta1, double beta2, int step, void* stream) {
    MF_CHECK_ARG(p0 && g0 && m0 && v0 && p1 && g1 && m1 && v1 && step >= 1);
    MF_CHECK_ARG(n0 > 0 && n1 > 0 && (n0 & 3) == 0 && (n1 & 3) == 0);
    MF_CHECK_ARG((((uintptr_t)p0 | (uintptr_t)g0 | (uintptr_t)m0 | (uintptr_t)v0 | (uintptr_t)p1 | (uintptr_t)g1 | (uintptr_t)m1 | (uintptr_t)v1) & 15) == 0);
    AdamTensor t0{(float4*)p0, (float4*)g0, (float4*)m0, (float4*)v0, n0 / 4, adam_scalars(lr0, beta1, beta2, eps0, wd0, step)};
    AdamTensor t1{(float4*)p1, (float4*)g1, (float4*)m1, (float4*)v1, n1 / 4, adam_scalars(lr1, beta1, beta2, eps1, wd1, step)};
    const int64_t cap = (int64_t)mf_sm_count_cached() * 8;
    const int64_t w0 = (t0.n4 + 255) / 256, w1 = (t1.n4 + 255) / 256;
    const int b0 = (int)(w0 < cap ? w0 : cap), b1 = (int)(w1 < 64 ? w1 : 64);
    adam_pair_kernel<<<(unsigned)(b0 + b1), 256, 0, (cudaStream_t)stream>>>(t0, t1, b0);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

MF_API int mf_adam_step_multi(int n_tensors, float* const* p, float* const* g, float* const* m, float* const* v,
                              const int64_t* n, double lr, double beta1, double beta2, double eps, double weight_decay,
                              int step, int zero_grad, void* stream) {
    MF_CHECK_ARG(n_tensors >= 0 && (n_tensors == 0 || (p && g && m && v && n)));
    for (int t = 0; t < n_tensors; ++t) {
        const int rc = mf_adam_step(p[t], g[t], m[t], v[t], n[t], lr, beta1, beta2, eps, weight_decay, step, zero_grad, stream);
        if (rc) return rc;
    }
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Uniform lattice (sampling_helper.py:38-48).
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline void lattice_params(int len, int num, int& step, int& start) {
    const int interval = (len - num) / (num + 1), offset = (len - num) % (num + 1);
    step = interval + 1; start = interval + offset / 2;
}

__global__ void lattice_kernel(int img_h, int img_w, int num_h, int num_w, int64_t* __restrict__ rows, int64_t* __restrict__ cols) {
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= num_h * num_w) return;
    int sh, oh, sw, ow;
    lattice_params(img_h, num_h, sh, oh);
    lattice_params(img_w, num_w, sw, ow);
    rows[t] = (int64_t)(t / num_w) * sh + oh;
    cols[t] = (int64_t)(t % num_w) * sw + ow;
}

MF_API int mf_sample_pixels_uniform(int img_h, int img_w, int num_h, int num_w, int64_t* rows, int64_t* cols, void* stream) {
    MF_CHECK_ARG(img_h > 0 && img_w > 0 && num_h > 0 && num_w > 0 && num_h <= img_h && num_w <= img_w && rows && cols);
    lattice_kernel<<<(num_h * num_w + 255) / 256, 256, 0, (cudaStream_t)stream>>>(img_h, img_w, num_h, num_w, rows, cols);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// ---------------------------------------------------------------------------------------------
// Top-k of keys*mask by (value descending, index ascending): torch.topk(samp_v, num)[1] with the
// tie rule made explicit (oracle/sampling.py).  Every element gets the distinct 64-bit key
//   key = (float_bits(v) << 32) | ~index        (v >= 0, so the bit pattern is order preserving)
// and the k largest keys are found by an MSB-first radix select (6 digit passes, each pass one
// kernel whose last-finishing block scans the histogram), then compacted and sorted by one CTA.
// ---------------------------------------------------------------------------------------------
constexpr int TOPK_MAX = 4096;
constexpr int RADIX_BINS = 2048;

struct TopkState {
    unsigned long long prefix;      // digits fixed so far (aligned to their bit position)
    unsigned long long mask;        // which bits of the key are fixed
    int k_rem;                      // how many keys are still to be taken at / below the prefix
    unsigned int done;              // block ticket of the current pass
    unsigned int n_sel;             // compaction cursor
    unsigned int hist[RADIX_BINS];
};

__device__ __forceinline__ unsigned long long topk_key(const float* __restrict__ depth, const float* __restrict__ keys,
                                                       int64_t i, int img_w, int lat_h, int lat_w, int sh, int oh, int sw, int ow) {
    float mask = depth[i] > 0.f ? 1.f : 0.f;
    if (lat_h > 0) {                                   // sample_pixels_mix: lattice pixels are excluded (:58)
        const int r = (int)(i / img_w), c = (int)(i % img_w);
        const int rr = r - oh, cc = c - ow;
        if (rr >= 0 && cc >= 0 && rr % sh == 0 && cc % sw == 0 && rr / sh < lat_h && cc / sw < lat_w) mask = 0.f;
    }
    const float v = __fmul_rn(mask, keys[i]);
    return ((unsigned long long)__float_as_uint(v) << 32) | (unsigned long long)(~(unsigned int)i);
}

__global__ void topk_init_kernel(TopkState* st, int k) {
    const int t = threadIdx.x + blockIdx.x * blockDim.x;
    if (t == 0) { st->prefix = 0ull; st->mask = 0ull; st->k_rem = k; st->done = 0u; st->n_sel = 0u; }
    if (t < RADIX_BINS) st->hist[t] = 0u;
}

__global__ void __launch_bounds__(256) topk_pass_kernel(const float* __restrict__ depth, const float* __restrict__ keys, int64_t n,
                                                        int img_w, int lat_h, int lat_w, int sh, int oh, int sw, int ow,
                                                        int shift, int bits, TopkState* st) {
    __shared__ unsigned int h[RADIX_BINS];
    __shared__ bool last;
    const int nb = 1 << bits;
    for (int b = threadIdx.x; b < nb; b += blockDim.x) h[b] = 0u;
    __syncthreads();
    const unsigned long long prefix = st->prefix, mask = st->mask;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long key = topk_key(depth, keys, i, img_w, lat_h, lat_w, sh, oh, sw, ow);
        if ((key & mask) == prefix) atomicAdd(&h[(unsigned int)(key >> shift) & (nb - 1)], 1u);
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nb; b += blockDim.x)
        if (h[b]) atomicAdd(&st->hist[b], h[b]);
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) last = (atomicAdd(&st->done, 1u) == gridDim.x - 1);
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last block: walk the histogram from the top digit down (single thread; <= 2048 bins)
    if (threadIdx.x == 0) {
        int k = st->k_rem, b = nb - 1;
        volatile unsigned int* gh = st->hist;
        for (; b > 0; --b) {
            const int c = (int)gh[b];
            if (c >= k) break;
            k -= c;
        }
        st->k_rem = k;
        st->prefix = prefix | ((unsigned long long)b << shift);
        st->mask = mask | ((unsigned long long)(nb - 1) << shift);
        st->done = 0u;
    }
    __syncthreads();
    for (int b = threadIdx.x; b < nb; b += blockDim.x) st->hist[b] = 0u;
}

__global__ void __launch_bounds__(256) topk_compact_kernel(const float* __restrict__ depth, const float* __restrict__ keys, int64_t n,
                                                           int img_w, int lat_h, int lat_w, int sh, int oh, int sw, int ow,
                                                           TopkState* st, unsigned long long* __restrict__ sel, int k) {
    const unsigned long long thr = st->prefix;        // after the last pass: the k-th largest key itself
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const unsigned long long key = topk_key(depth, keys, i, img_w, lat_h, lat_w, sh, oh, sw, ow);
        if (key >= thr) {
            const unsigned int slot = atomicAdd(&st->n_sel, 1u);
            if (slot < (unsigned int)k) sel[slot] = key;
        }
    }
}

// One CTA: bitonic sort (descending) of the k selected keys, then decode the indices.
__global__ void __launch_bounds__(1024) topk_sort_kernel(const unsigned long long* __restrict__ sel, int k, int img_w,
                                                         int n_lat, int64_t* __restrict__ indices, int64_t* __restrict__ rows,
                                                         int64_t* __restrict__ cols) {
    __shared__ unsigned long long s[TOPK_MAX];
    int np2 = 1;
    while (np2 < k) np2 <<= 1;
    for (int i = threadIdx.x; i < np2; i += blockDim.x) s[i] = i < k ? sel[i] : 0ull;
    __syncthreads();
    for (int size = 2; size <= np2; size <<= 1)
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < np2; i += blockDim.x) {
                const int j = i ^ stride;
                if (j > i) {
                    const bool desc = (i & size) == 0;
                    const unsigned long long a = s[i], b = s[j];
                    if (desc ? (a < b) : (a > b)) { s[i] = b; s[j] = a; }
                }
            }
            __syncthreads();
        }
    for (int i = threadIdx.x; i < k; i += blockDim.x) {
        const int64_t idx = (int64_t)(~(unsigned int)(s[i] & 0xffffffffull));
        if (indices) indices[i] = idx;
        if (rows) { rows[n_lat + i] = idx / img_w; cols[n_lat + i] = idx % img_w; }
    }
}

MF_API int64_t mf_topk_workspace_size(int64_t n) { (void)n; return (int64_t)sizeof(TopkState) + TOPK_MAX * sizeof(unsigned long long) + 256; }

MF_API int mf_sample_pixels_topk(const float* depth, const float* keys, int img_h, int img_w, int lattice_h, int lattice_w, int num,
                                 int64_t* indices, int64_t* rows, int64_t* cols, void* workspace, void* stream) {
    MF_CHECK_ARG(depth && keys && workspace && img_h > 0 && img_w > 0);
    MF_CHECK_ARG((lattice_h > 0) == (lattice_w > 0));
    MF_CHECK_ARG((rows == nullptr) == (cols == nullptr));
    const int n_lat = lattice_h * lattice_w;
    const int k = num - n_lat;
    const int64_t n = (int64_t)img_h * img_w;
    MF_CHECK_ARG(k >= 0 && k <= TOPK_MAX && k <= n);
    MF_CHECK_ARG(n < (1ll << 32));
    MF_CHECK_ARG(lattice_h == 0 || (rows && lattice_h <= img_h && lattice_w <= img_w));
    MF_CHECK_ARG(indices || rows);
    cudaStream_t st = (cudaStream_t)stream;
    int sh = 1, oh = 0, sw = 1, ow = 0;
    if (n_lat > 0) {
        lattice_params(img_h, lattice_h, sh, oh);
        lattice_params(img_w, lattice_w, sw, ow);
        lattice_kernel<<<(n_lat + 255) / 256, 256, 0, st>>>(img_h, img_w, lattice_h, lattice_w, rows, cols);
        MF_LAUNCH_CHECK();
    }
    if (k == 0) return MF_OK;
    TopkState* state = (TopkState*)workspace;
    unsigned long long* sel = (unsigned long long*)((char*)workspace + ((sizeof(TopkState) + 255) / 256) * 256);
    topk_init_kernel<<<(RADIX_BINS + 255) / 256, 256, 0, st>>>(state, k);
    MF_LAUNCH_CHECK();
    const int64_t want = (n + 255) / 256;
    const unsigned blocks = (unsigned)(want < 2 * mf_sm_count_cached() ? want : 2 * mf_sm_count_cached());
    const int shifts[6] = {53, 42, 32, 21, 10, 0}, nbits[6] = {11, 11, 10, 11, 11, 10};
    for (int p = 0; p < 6; ++p) {
        topk_pass_kernel<<<blocks, 256, 0, st>>>(depth, keys, n, img_w, lattice_h, lattice_w, sh, oh, sw, ow, shifts[p], nbits[p], state);
        MF_LAUNCH_CHECK();
    }
    topk_compact_kernel<<<blocks, 256, 0, st>>>(depth, keys, n, img_w, lattice_h, lattice_w, sh, oh, sw, ow, state, sel, k);
    MF_LAUNCH_CHECK();
    topk_sort_kernel<<<1, 1024, 0, st>>>(sel, k, img_w, n_lat, indices, rows, cols);
    MF_LAUNCH_CHECK();
    return MF_OK;
}


// ---------------------------------------------------------------------------------------------
// N1: keyframe ray store on the device (model/keyframeSet.py:25,76-79,170-175,386-455).
// store (num_kf, n_rays, 7) fp32 = [dir_cam | rgb | depth] of the lattice-downsampled keyframes.
// ---------------------------------------------------------------------------------------------
// add_keyframe: rows of the full-resolution frame picked by the uniform lattice (pixel index = row * W + col)
__global__ void kf_store_kernel(const float* __restrict__ dirs, const float* __restrict__ rgb, const float* __restrict__ depth,
                                const int64_t* __restrict__ rows, const int64_t* __restrict__ cols, int img_w, int64_t n_rays,
                                float* __restrict__ slot) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_rays) return;
    const int64_t px = rows[j] * img_w + cols[j];
    float* o = slot + j * 7;
    o[0] = dirs[px * 3]; o[1] = dirs[px * 3 + 1]; o[2] = dirs[px * 3 + 2];
    o[3] = rgb[px * 3]; o[4] = rgb[px * 3 + 1]; o[5] = rgb[px * 3 + 2];
    o[6] = depth[px];
}

MF_API int mf_kf_store(const float* dirs_cam, const float* rgb, const float* depth, const int64_t* rows, const int64_t* cols,
                       int img_w, int64_t n_rays, float* store_slot, void* stream) {
    MF_CHECK_ARG(n_rays >= 0 && img_w > 0);
    if (n_rays == 0) return MF_OK;
    MF_CHECK_ARG(dirs_cam && rgb && depth && rows && cols && store_slot);
    kf_store_kernel<<<(unsigned)((n_rays + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dirs_cam, rgb, depth, rows, cols, img_w, n_rays, store_slot);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// sample_rays_in_submap (model/keyframeSet.py:386-437) for given index draws: output ray j comes from
//   j <  n_first                : keyframe first_kf_id, ray idx_first[j]               -> kf_index 0
//   j <  n_first + n_other      : idx = idx_other[.]: keyframe other_ids[idx / n_rays], ray idx % n_rays -> kf_index idx / n_rays + 1
//   else                        : keyframe last_kf_id, ray idx_last[.]                 -> kf_index n_related - 1
// other_ids = related_kf_ids + 1 (n_other_kf entries).  Integer outputs are exactly the reference's.
__global__ void kf_gather_kernel(const float* __restrict__ store, int64_t n_rays, int64_t first_kf_id,
                                 const int64_t* __restrict__ other_ids, int64_t last_kf_id, int n_related,
                                 const int64_t* __restrict__ idx_first, int64_t n_first, const int64_t* __restrict__ idx_other,
                                 int64_t n_other, const int64_t* __restrict__ idx_last, int64_t n_last,
                                 float* __restrict__ out, int64_t* __restrict__ kf_ids, int64_t* __restrict__ kf_indices) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_first + n_other + n_last) return;
    int64_t kf, ray, kidx;
    if (j < n_first) { kf = first_kf_id; ray = idx_first[j]; kidx = 0; }
    else if (j < n_first + n_other) {
        const int64_t idx = idx_other[j - n_first], local = idx / n_rays;
        kf = other_ids[local]; ray = idx - local * n_rays; kidx = local + 1;
    } else { kf = last_kf_id; ray = idx_last[j - n_first - n_other]; kidx = n_related - 1; }
    const float* src = store + (kf * n_rays + ray) * 7;
    float* o = out + j * 7;
#pragma unroll
    for (int k = 0; k < 7; ++k) o[k] = src[k];
    kf_ids[j] = kf; kf_indices[j] = kidx;
}

MF_API int mf_kf_gather_rays(const float* store, int64_t n_rays, int64_t first_kf_id, const int64_t* other_kf_ids,
                             int64_t last_kf_id, int n_related, const int64_t* idx_first, int64_t n_first,
                             const int64_t* idx_other, int64_t n_other, const int64_t* idx_last, int64_t n_last,
                             float* out_rays7, int64_t* out_kf_ids, int64_t* out_kf_indices, void* stream) {
    MF_CHECK_ARG(n_rays > 0 && n_related >= 1 && n_first >= 0 && n_other >= 0 && n_last >= 0);
    const int64_t n = n_first + n_other + n_last;
    if (n == 0) return MF_OK;
    MF_CHECK_ARG(store && out_rays7 && out_kf_ids && out_kf_indices);
    MF_CHECK_ARG((n_first == 0 || idx_first) && (n_other == 0 || (idx_other && other_kf_ids)) && (n_last == 0 || idx_last));
    kf_gather_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(store, n_rays, first_kf_id, other_kf_ids, last_kf_id,
                                                                                  n_related, idx_first, n_first, idx_other, n_other,
                                                                                  idx_last, n_last, out_rays7, out_kf_ids, out_kf_indices);
    MF_LAUNCH_CHECK();
    return MF_OK;
}


// ---------------------------------------------------------------------------------------------
// Sampling without replacement on the device (python random.sample(range(n), k) in the reference): element j of the
// sample is perm(j), where perm is a keyed pseudo-random PERMUTATION of [0, n): a 4-round balanced Feistel network on
// 2b bits (4^b >= n) with cycle walking.  O(k) work, no sort, k distinct values by construction; oracle/keyframes.py
// restates it in numpy (bit-exact).  mix32 = the public-domain "lowbias32" integer hash.
// ---------------------------------------------------------------------------------------------
__host__ __device__ inline uint32_t mf_mix32(uint32_t x) {
    x ^= x >> 16; x *= 0x7feb352dU; x ^= x >> 15; x *= 0x846ca68bU; x ^= x >> 16;
    return x;
}
__host__ __device__ inline int mf_feistel_half_bits(uint64_t n) {
    int b = 1;
    while (((uint64_t)1 << (2 * b)) < n) ++b;
    return b;
}
__host__ __device__ inline uint64_t mf_feistel_perm(uint64_t j, uint64_t n, int b, uint32_t seed) {
    const uint32_t mask = (uint32_t)(((uint64_t)1 << b) - 1);
    uint64_t x = j;
    do {
        uint32_t l = (uint32_t)(x >> b) & mask, r = (uint32_t)x & mask;
#pragma unroll
        for (int round = 0; round < 4; ++round) {
            const uint32_t key = mf_mix32(seed + 0x9e3779b9U * (uint32_t)(round + 1));
            const uint32_t t = l ^ (mf_mix32(r ^ key) & mask);
            l = r; r = t;
        }
        x = ((uint64_t)l << b) | r;
    } while (x >= n);
    return x;
}

__global__ void sample_distinct_kernel(int64_t n, int64_t k, uint32_t seed, int64_t* __restrict__ out) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= k) return;
    out[j] = (int64_t)mf_feistel_perm((uint64_t)j, (uint64_t)n, mf_feistel_half_bits((uint64_t)n), seed);
}

MF_API int mf_sample_distinct(int64_t n, int64_t k, uint32_t seed, int64_t* out, void* stream) {
    MF_CHECK_ARG(n >= 1 && k >= 0 && k <= n && n <= ((int64_t)1 << 40));
    if (k == 0) return MF_OK;
    MF_CHECK_ARG(out);
    sample_distinct_kernel<<<(unsigned)((k + 255) / 256), 256, 0, (cudaStream_t)stream>>>(n, k, seed, out);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// sample_rays_in_submap with the draws made in the kernel: segment s uses seed + s (first, other, last)
__global__ void kf_sample_kernel(const float* __restrict__ store, int64_t n_rays, int64_t first_kf_id,
                                 const int64_t* __restrict__ other_ids, int64_t n_other_kf, int64_t last_kf_id, int n_related,
                                 int64_t n_first, int64_t n_other, int64_t n_last, uint32_t seed,
                                 float* __restrict__ out, int64_t* __restrict__ kf_ids, int64_t* __restrict__ kf_indices,
                                 int64_t* __restrict__ out_idx) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_first + n_other + n_last) return;
    int64_t kf, ray, kidx, idx;
    if (j < n_first) {
        idx = (int64_t)mf_feistel_perm((uint64_t)j, (uint64_t)n_rays, mf_feistel_half_bits((uint64_t)n_rays), seed);
        kf = first_kf_id; ray = idx; kidx = 0;
    } else if (j < n_first + n_other) {
        const uint64_t pop = (uint64_t)(n_other_kf * n_rays);
        idx = (int64_t)mf_feistel_perm((uint64_t)(j - n_first), pop, mf_feistel_half_bits(pop), seed + 1u);
        const int64_t local = idx / n_rays;
        kf = other_ids[local]; ray = idx - local * n_rays; kidx = local + 1;
    } else {
        idx = (int64_t)mf_feistel_perm((uint64_t)(j - n_first - n_other), (uint64_t)n_rays, mf_feistel_half_bits((uint64_t)n_rays), seed + 2u);
        kf = last_kf_id; ray = idx; kidx = n_related - 1;
    }
    const float* src = store + (kf * n_rays + ray) * 7;
    float* o = out + j * 7;
#pragma unroll
    for (int k = 0; k < 7; ++k) o[k] = src[k];
    kf_ids[j] = kf; kf_indices[j] = kidx;
    if (out_idx) out_idx[j] = idx;
}

MF_API int mf_kf_sample_rays(const float* store, int64_t n_rays, int64_t first_kf_id, const int64_t* other_kf_ids, int64_t n_other_kf,
                             int64_t last_kf_id, int n_related, int64_t n_first, int64_t n_other, int64_t n_last, uint32_t seed,
                             float* out_rays7, int64_t* out_kf_ids, int64_t* out_kf_indices, int64_t* out_idx, void* stream) {
    MF_CHECK_ARG(n_rays > 0 && n_related >= 1 && n_first >= 0 && n_other >= 0 && n_last >= 0 && n_other_kf >= 0);
    MF_CHECK_ARG(n_first <= n_rays && n_last <= n_rays && n_other <= n_other_kf * n_rays);
    const int64_t n = n_first + n_other + n_last;
    if (n == 0) return MF_OK;
    MF_CHECK_ARG(store && out_rays7 && out_kf_ids && out_kf_indices && (n_other == 0 || other_kf_ids));
    kf_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(store, n_rays, first_kf_id, other_kf_ids, n_other_kf,
                                                                                  last_kf_id, n_related, n_first, n_other, n_last, seed,
                                                                                  out_rays7, out_kf_ids, out_kf_indices, out_idx);
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// The mapping batch of submap initialisation (first_frame_mapping / initialize_new_localMLP, mipsfusion.py:135-138,178,209):
// random.sample(range(H*W), n) drawn as perm(j) inside the gather, decoded column-major (h = i % H, w = i / H) as the
// reference indexes its (H, W) frame, and [dir | rgb | depth] of pixel (h, w) written to ray j.  idx: explicit draws instead.
__global__ void frame_sample_kernel(const float* __restrict__ dirs, const float* __restrict__ rgb, const float* __restrict__ depth,
                                    int img_h, int img_w, int64_t n, uint32_t seed, int half_bits, const int64_t* __restrict__ idx,
                                    float* __restrict__ out, int64_t* __restrict__ out_idx) {
    const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    const int64_t i = idx ? idx[j] : (int64_t)mf_feistel_perm((uint64_t)j, (uint64_t)img_h * img_w, half_bits, seed);
    const int64_t h = i % img_h, w = i / img_h;
    const int64_t px = h * img_w + w;
    float* o = out + j * 7;
    o[0] = dirs[px * 3]; o[1] = dirs[px * 3 + 1]; o[2] = dirs[px * 3 + 2];
    o[3] = rgb[px * 3]; o[4] = rgb[px * 3 + 1]; o[5] = rgb[px * 3 + 2];
    o[6] = depth[px];
    if (out_idx) out_idx[j] = i;
}

MF_API int mf_frame_sample_rays(const float* dirs_cam, const float* rgb, const float* depth, int img_h, int img_w, int64_t n,
                                uint32_t seed, const int64_t* idx, float* out_rays7, int64_t* out_idx, void* stream) {
    MF_CHECK_ARG(img_h > 0 && img_w > 0 && n >= 0 && n <= (int64_t)img_h * img_w);
    if (n == 0) return MF_OK;
    MF_CHECK_ARG(dirs_cam && rgb && depth && out_rays7);
    const int half_bits = mf_feistel_half_bits((uint64_t)img_h * img_w);
    frame_sample_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(dirs_cam, rgb, depth, img_h, img_w, n, seed,
                                                                                     half_bits, idx, out_rays7, out_idx);
    MF_LAUNCH_CHECK();
    return MF_OK;
}
