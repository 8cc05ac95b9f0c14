// Tensor-core forward, producer / consumer version (the default): one persistent CTA per SM, 16 warps.
//
//   warps 0-7  PRODUCERS  encode 128-point tiles: coordinates, 48 sines, the 128 table gathers per point (the
//                         load/store unit is the bound of this stage: one gather lane per cycle), bf16 hi/lo
//                         split, and write the operand words with tcgen05.st straight into a STAGING region of
//                         tensor memory (two stages, 96 columns each) -- tensor memory is the ring buffer, no
//                         shared-memory staging of activations.
//   warps 8-15 CONSUMERS  run the decoder on the staged tile: the layer-1 MMAs read the encoded inputs and the
//                         layer-3 MMAs the grid features directly from the staging columns; activations live in
//                         the consumer's own operand region; epilogues, narrow heads and the store as before.
//
// The two roles only meet at two mbarrier pairs: full[s] (256 producer arrivals: operand words of stage s are in
// tensor memory) and empty[s] (tcgen05.commit of the layer-3 MMAs: stage s has been consumed).  While the
// producers wait on memory the consumers own the issue slots, and vice versa: the gather stage and the decoder
// overlap instead of alternating.
//
// Tensor memory (512 columns allocated): D [0,128) | A_hi [128,192) | A_lo [192,256) |
//   stage s at 256 + 96 s: e_hi [0,32) e_lo [32,64) g_hi [64,80) g_lo [80,96).
#pragma once
#include "field_tc.cuh"

constexpr int T3_GT = 256;                       // threads per role
constexpr int T3_D = 0, T3_A_HI = 128, T3_A_LO = 192, T3_STG = 256, T3_STG_COLS = 96;
constexpr int T3_E_HI = 0, T3_E_LO = 32, T3_G_HI = 64, T3_G_LO = 80;
constexpr int T3_CPART_ROWS = 6;                 // colour head, e part: 2 half-point partials x 3 channels, per stage
constexpr int T3_PART_ROWS = 13;                 // consumer: 3 colour-emb partials + 2 x 5 logit partials
constexpr int T3S_CPART = ((IMG_BYTES + 127) / 128) * 128;
constexpr int T3S_PART = T3S_CPART + 2 * T3_CPART_ROWS * TC_LD * 4;
constexpr int T3S_OUT = T3S_PART + T3_PART_ROWS * TC_LD * 4;
constexpr int T3S_BAR = T3S_OUT + MF_RAW_DIM * TC_LD * 4;
constexpr size_t SMEM_TC3 = T3S_BAR + 64 + 1024;                 // bars [0,5) | tile queue at +40 | image barrier [7] at +56
static_assert(SMEM_TC3 <= 227 * 1024, "shared memory budget");

__device__ __forceinline__ void t3_cons_sync() { asm volatile("bar.sync 1, %0;" ::"n"(T3_GT) : "memory"); }

struct T3Cons {
    uint8_t* img; const float* fw; float* part; float* out; uint64_t* bar;
    uint32_t tmem, lane_base, phase;
    int tid;
    bool ok;
};

// one decoder layer on the consumer side; a_col(ks, lo) = tensor-memory column (relative to the allocation) of k-step ks.
// The issue loop is fully unrolled and the weight descriptors are one base descriptor plus constants (start-address field in
// 16-byte units): the 255 other consumer threads wait while thread 0 issues, so its instruction count is on the tile's critical path.
template <int KS, int N_OUT = 128, class ColFn, class AfterFn>
__device__ __forceinline__ void t3_run_layer(T3Cons& c, int img_hi, int img_lo, ColFn a_col, AfterFn after_issue) {
    umma::wait_st();
    umma::fence_before_sync();
    t3_cons_sync();
    if (c.tid == 0) {
        umma::fence_after_sync();
        constexpr uint32_t idesc = umma::idesc_bf16(128, N_OUT, 0, 0);     // N_OUT < 128: only the first N_OUT output features
        const uint64_t dh = umma::smem_desc_sw128(umma::smem_u32(c.img + img_hi), 16, 1024);
        const uint64_t dl = umma::smem_desc_sw128(umma::smem_u32(c.img + img_lo), 16, 1024);
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
#pragma unroll
            for (int ks = 0; ks < KS; ++ks) {
                const uint32_t off = (uint32_t)(((ks >> 2) * IMG_BLOCK + (ks & 3) * 32) >> 4);
                umma::mma_ts(c.tmem + T3_D, c.tmem + (uint32_t)a_col(ks, pass == 2), (pass == 1 ? dl : dh) + off, idesc, (pass | ks) ? 1u : 0u);
            }
        }
        umma::commit(c.bar);
        after_issue();
    }
    c.ok &= umma::mbar_wait(c.bar, c.phase);
    c.phase ^= 1;
    umma::fence_after_sync();
}

__device__ __forceinline__ void t3_load32(const T3Cons& c, int col, float (&v)[32]) {
    uint32_t r[32];
    umma::tmem_ld32(c.lane_base + (uint32_t)col, r);
    umma::wait_ld();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void t3_store32(const T3Cons& c, int f0, const float (&v)[32]) {
    uint32_t hi[16], lo[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) umma::split2(v[2 * i], v[2 * i + 1], hi[i], lo[i]);
    umma::tmem_st16(c.lane_base + (uint32_t)(T3_A_HI + f0 / 2), hi);
    umma::tmem_st16(c.lane_base + (uint32_t)(T3_A_LO + f0 / 2), lo);
}

template <class Src, class Epi, bool SDF_ONLY>
__global__ void __launch_bounds__(2 * T3_GT, 1) field_fwd_tc3_kernel(FieldDev f, Src src, Epi epi, int64_t N,
                                                                     const unsigned int* __restrict__ n_dev,
                                                                     const uint8_t* __restrict__ img, int* __restrict__ err,
                                                                     long long* __restrict__ prof, int* __restrict__ tile_ctr = nullptr) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ uint32_t tmem_ptr_s;
    // profiling stamps (mf_debug_profile): CTA 0, third tile; producers -> prof[40..], consumers -> prof[48..]
#define T3_MARK(slot) do { if (prof && blockIdx.x == 0 && tid == 0 && k == 2) prof[slot] = clock64(); } while (0)
    mf_pdl_wait();                                       // (programmatic launch, mf_common.cuh: no global access before it)
    if (n_dev) N = (int64_t)*n_dev;
    if (prof && blockIdx.x == 0 && threadIdx.x == 0) prof[29] = clock64();
    if (prof && threadIdx.x == 0 && blockIdx.x < 256) prof[64 + 2 * blockIdx.x] = mf_globaltimer();
    uint8_t* base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    uint64_t* bars = (uint64_t*)(base + T3S_BAR);            // [0] mma, [1,2] full, [3,4] empty
    if ((threadIdx.x >> 5) == 0) umma::tmem_alloc<512>(&tmem_ptr_s);
    if (threadIdx.x == 0) {
        umma::mbar_init(bars + 0, 1);
        umma::mbar_init(bars + 1, T3_GT); umma::mbar_init(bars + 2, T3_GT);
        umma::mbar_init(bars + 3, 1); umma::mbar_init(bars + 4, 1);
        umma::mbar_init(bars + 7, 1);
        umma::fence_barrier_init();
        // the weight image (166 KB) comes in through the bulk-copy engine while the CTA sets up (a copy loop over all threads
        // took ~20 dependent L2 round trips per thread)
        constexpr uint32_t CHUNK = 32768;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(umma::smem_u32(bars + 7)), "r"((uint32_t)IMG_BYTES) : "memory");
        for (uint32_t off = 0; off < (uint32_t)IMG_BYTES; off += CHUNK) {
            const uint32_t nb = (uint32_t)IMG_BYTES - off < CHUNK ? (uint32_t)IMG_BYTES - off : CHUNK;
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(umma::smem_u32(base + off)), "l"(img + off), "r"(nb), "r"(umma::smem_u32(bars + 7)) : "memory");
        }
    }
    umma::fence_before_sync();
    __syncthreads();
    umma::fence_after_sync();
    bool img_ok = umma::mbar_wait(bars + 7, 0);            // the image has landed (visible to this thread and to the tensor core)
    const uint32_t tmem = tmem_ptr_s;
    const bool producer = threadIdx.x < T3_GT;
    const int tid = threadIdx.x & (T3_GT - 1), p = tid & 127, h = tid >> 7;
    const uint32_t lane_base = tmem + ((uint32_t)(((tid >> 5) & 3) * 32) << 16);
    const float* fw = (const float*)(base + IMG_F32);
    const int64_t n_tiles = (N + TC_TP - 1) / TC_TP;
    bool ok = img_ok;
    // Tile queue.  The first two tiles of a CTA are static (blockIdx.x, blockIdx.x + gridDim.x); from the third on an elected
    // producer thread draws the tile of iteration k + 2 from a global counter while it works on iteration k and leaves it in
    // tq[(k + 2) & 3] (tile_ctr == NULL: static striding through the same queue).  SMs do not run this kernel at the same
    // speed -- measured CTA lifetimes at C1 with static striding: 124 .. 163 us (scripts/prof_cta.py) -- so the fast ones take
    // more tiles.  Which CTA evaluates a tile does not change any result.
    volatile int* tq = reinterpret_cast<volatile int*>(base + T3S_BAR + 40);
    if (threadIdx.x < 4) tq[threadIdx.x] = 0;              // (before the first rendezvous below; speculative reads see a valid tile)

    if (producer) {
        // =========================== producers: encode into the staging columns ===========================
        const float2* grid2 = reinterpret_cast<const float2*>(f.grid);
        for (uint32_t k = 0;; ++k) {
            const int s = (int)(k & 1u);
            const uint32_t stg = lane_base + (uint32_t)(T3_STG + T3_STG_COLS * s);
            float* cpart = (float*)(base + T3S_CPART) + s * T3_CPART_ROWS * TC_LD;
            T3_MARK(40);
            if (prof && blockIdx.x == 0 && tid == 0 && k < 12) prof[16 + k] = clock64();      // per-tile start stamps
            // The point is loaded BEFORE the wait below (its latency hides behind it), from a speculative read of the tile queue:
            // the entry was written a whole tile period ago, but only the wait orders this thread after that write -- so the entry
            // is read again afterwards and the point reloaded in the (never observed) case that the two reads differ.
            const int64_t tile_e = k < 2 ? (int64_t)blockIdx.x + (int64_t)k * gridDim.x : (int64_t)tq[k & 3u];
            float x[3] = {0.f, 0.f, 0.f};
            if (tile_e >= 0 && tile_e < n_tiles && tile_e * TC_TP + p < N) src.point(tile_e * TC_TP + p, f, x);
            // stage s is free once the layer-3 MMAs of the tile that used it two tiles ago have completed
            ok &= umma::mbar_wait(bars + 3 + s, ((k >> 1) & 1u) ^ 1u);
            umma::fence_after_sync();
            const int64_t tile = k < 2 ? tile_e : (int64_t)tq[k & 3u];
            if (tile >= n_tiles) break;
            if (tid == 0) {                                // publish the tile of iteration k + 2 (see the tile queue note above)
                const int64_t t2 = tile_ctr ? 2 * (int64_t)gridDim.x + atomicAdd(tile_ctr, 1) : tile + 2 * (int64_t)gridDim.x;
                tq[(k + 2u) & 3u] = (int)(t2 < n_tiles ? t2 : n_tiles);
            }
            const int64_t i = tile * TC_TP + p;
            const bool valid = i < N;
            if (tile != tile_e) {
                x[0] = x[1] = x[2] = 0.f;
                if (valid) src.point(i, f, x);
            }
            T3_MARK(41);
            // ---- frequency features: this thread owns slot groups 2h, 2h+1 ----
            float r[3] = {0.f, 0.f, 0.f};
#pragma unroll
            for (int sg = 0; sg < 2; ++sg) {
                const int qq = 2 * h + sg;
                float e[16];
#pragma unroll
                for (int jj = 0; jj < 12; ++jj) {
                    const int j = qq * 12 + jj, d = j >> 4, kk = (j & 15) >> 1, ph = j & 1;
                    e[jj] = sin_reduced(freq_arg(x[d], kk, ph));
                }
                e[12] = qq == 0 ? x[0] : 0.f; e[13] = qq == 0 ? x[1] : 0.f; e[14] = qq == 0 ? x[2] : 0.f; e[15] = 0.f;
                uint32_t hi[8], lo[8];
#pragma unroll
                for (int t = 0; t < 8; ++t) umma::split2(e[2 * t], e[2 * t + 1], hi[t], lo[t]);
                umma::tmem_st8(stg + T3_E_HI + 8 * qq, hi);
                umma::tmem_st8(stg + T3_E_LO + 8 * qq, lo);
                if (f.feat) {
                    uint32_t* fo = f.feat + (size_t)tile * FEAT_TILE_WORDS + (size_t)qq * FEAT_WORDS * TC_TP + p;
#pragma unroll
                    for (int t = 0; t < 8; ++t) { fo[t * TC_TP] = hi[t]; fo[(8 + t) * TC_TP] = lo[t]; }
                }
                if (!SDF_ONLY) {
                    const float* wre = fw + F_WR_E + 16 * qq;
#pragma unroll
                    for (int t = 0; t < 16; ++t)
#pragma unroll
                        for (int ch = 0; ch < 3; ++ch) r[ch] = fmaf(wre[ch * 64 + t], e[t], r[ch]);
                }
            }
            if (!SDF_ONLY) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) cpart[(h * 3 + ch) * TC_LD + p] = r[ch];
            }
            T3_MARK(42);
            // ---- grid features: levels [8h, 8h+8) ----
            // (rolled loops: the two roles run different code at the same time, so instruction-cache footprint matters)
#pragma unroll 1
            for (int sg = 0; sg < 2; ++sg) {
                float gf[8];
#pragma unroll 2
                for (int ll = 0; ll < 4; ++ll) {
                    float2 v2 = make_float2(0.f, 0.f);
                    if (valid) v2 = grid_level_fwd(x, grid2, level_info(f, 8 * h + 4 * sg + ll), nullptr);
                    gf[2 * ll] = v2.x; gf[2 * ll + 1] = v2.y;
                }
                uint32_t ghi[4], glo[4];
#pragma unroll
                for (int t = 0; t < 4; ++t) umma::split2(gf[2 * t], gf[2 * t + 1], ghi[t], glo[t]);
                umma::tmem_st4(stg + T3_G_HI + 8 * h + 4 * sg, ghi);
                umma::tmem_st4(stg + T3_G_LO + 8 * h + 4 * sg, glo);
                if (f.feat) {
                    uint32_t* fo = f.feat + (size_t)tile * FEAT_TILE_WORDS + (size_t)(2 * h + sg) * FEAT_WORDS * TC_TP + p;
#pragma unroll
                    for (int t = 0; t < 4; ++t) { fo[(16 + t) * TC_TP] = ghi[t]; fo[(20 + t) * TC_TP] = glo[t]; }
                }
            }
            T3_MARK(43);
            umma::wait_st();
            umma::fence_before_sync();
            umma::mbar_arrive(bars + 1 + s);
            T3_MARK(44);
        }
    } else {
        // =========================== consumers: decoder on the staged tile ===========================
        T3Cons c;
        c.img = base; c.fw = fw; c.part = (float*)(base + T3S_PART); c.out = (float*)(base + T3S_OUT); c.bar = bars;
        c.tmem = tmem; c.lane_base = lane_base; c.phase = 0; c.tid = tid; c.ok = ok;
        float v[32];
        for (uint32_t k = 0;; ++k) {
            // (the queue entry of iteration k was written before the producers handed over tile k - 2, which this role has waited for)
            const int64_t tile = k < 2 ? (int64_t)blockIdx.x + (int64_t)k * gridDim.x : (int64_t)tq[k & 3u];
            if (tile >= n_tiles) break;
            const int s = (int)(k & 1u);
            const int stg = T3_STG + T3_STG_COLS * s;
            const float* cpart = (const float*)(base + T3S_CPART) + s * T3_CPART_ROWS * TC_LD;
            T3_MARK(48);
            c.ok &= umma::mbar_wait(bars + 1 + s, (k >> 1) & 1u);
            umma::fence_after_sync();
            T3_MARK(49);
            float rgb_e[3] = {0.f, 0.f, 0.f};
            if (!SDF_ONLY && h == 0) {
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) rgb_e[ch] = cpart[ch * TC_LD + p] + cpart[(3 + ch) * TC_LD + p];
            }
            // ---- pts_linear.0 + ReLU (A = staged e) ----
            t3_run_layer<4>(c, IMG_W1_HI, IMG_W1_LO, [stg](int ks, bool lo) { return stg + (lo ? T3_E_LO : T3_E_HI) + 8 * ks; }, []() {});
            T3_MARK(50);
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                const int f0 = 64 * h + 32 * half;
                t3_load32(c, T3_D + f0, v);
                const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_B1 + f0);
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 b = b4[k4];
                    v[4 * k4] = fmaxf(v[4 * k4] + b.x, 0.f); v[4 * k4 + 1] = fmaxf(v[4 * k4 + 1] + b.y, 0.f);
                    v[4 * k4 + 2] = fmaxf(v[4 * k4 + 2] + b.z, 0.f); v[4 * k4 + 3] = fmaxf(v[4 * k4 + 3] + b.w, 0.f);
                }
                t3_store32(c, f0, v);
            }
            T3_MARK(51);
            // ---- pts_linear.2 (SDF only: just the 64 sdf_emb outputs, 32 per thread) ----
            if (SDF_ONLY) {
                t3_run_layer<8, 64>(c, IMG_W2_HI, IMG_W2_LO, [](int ks, bool lo) { return (lo ? T3_A_LO : T3_A_HI) + 8 * ks; }, []() {});
                T3_MARK(52);
                const int f0 = 32 * h;
                t3_load32(c, T3_D + f0, v);
                const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_B2 + f0);
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 b = b4[k4];
                    v[4 * k4] += b.x; v[4 * k4 + 1] += b.y; v[4 * k4 + 2] += b.z; v[4 * k4 + 3] += b.w;
                }
                t3_store32(c, f0, v);
            } else {
            t3_run_layer<8>(c, IMG_W2_HI, IMG_W2_LO, [](int ks, bool lo) { return (lo ? T3_A_LO : T3_A_HI) + 8 * ks; }, []() {});
            T3_MARK(52);
            {
                float r[3] = {0.f, 0.f, 0.f};
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    const int f0 = 64 * h + 32 * half;
                    t3_load32(c, T3_D + f0, v);
                    const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_B2 + f0);
#pragma unroll
                    for (int k4 = 0; k4 < 8; ++k4) {
                        const float4 b = b4[k4];
                        v[4 * k4] += b.x; v[4 * k4 + 1] += b.y; v[4 * k4 + 2] += b.z; v[4 * k4 + 3] += b.w;
                    }
                    if (h == 0) {
                        t3_store32(c, f0, v);                    // sdf_emb -> features [0,64) of the layer-3 operand
                    } else {
#pragma unroll
                        for (int ch = 0; ch < 3; ++ch) {
                            const float4* w4 = reinterpret_cast<const float4*>(c.fw + F_WR_EMB + ch * 64 + 32 * half);
#pragma unroll
                            for (int k4 = 0; k4 < 8; ++k4) {
                                const float4 w = w4[k4];
                                r[ch] = fmaf(w.x, v[4 * k4], r[ch]); r[ch] = fmaf(w.y, v[4 * k4 + 1], r[ch]);
                                r[ch] = fmaf(w.z, v[4 * k4 + 2], r[ch]); r[ch] = fmaf(w.w, v[4 * k4 + 3], r[ch]);
                            }
                        }
                    }
                }
                if (h == 1) {
#pragma unroll
                    for (int ch = 0; ch < 3; ++ch) c.part[ch * TC_LD + p] = r[ch];
                }
            }
            }
            T3_MARK(53);
            // ---- sdf_linear.0 + ReLU (k-steps 0-3: sdf_emb, 4-5: staged grid features); releases the stage ----
            uint64_t* empty = bars + 3 + s;
            t3_run_layer<6>(c, IMG_W3_HI, IMG_W3_LO,
                         [stg](int ks, bool lo) { return ks < 4 ? (lo ? T3_A_LO : T3_A_HI) + 8 * ks : stg + (lo ? T3_G_LO : T3_G_HI) + 8 * (ks - 4); },
                         [empty]() { umma::commit(empty); });
            T3_MARK(54);
            {
                float sl[N_CLASS] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
                for (int half = 0; half < 2; ++half) {
                    const int f0 = 64 * h + 32 * half;
                    t3_load32(c, T3_D + f0, v);
                    const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_BS1 + f0);
#pragma unroll
                    for (int k4 = 0; k4 < 8; ++k4) {
                        const float4 b = b4[k4];
                        v[4 * k4] = fmaxf(v[4 * k4] + b.x, 0.f); v[4 * k4 + 1] = fmaxf(v[4 * k4 + 1] + b.y, 0.f);
                        v[4 * k4 + 2] = fmaxf(v[4 * k4 + 2] + b.z, 0.f); v[4 * k4 + 3] = fmaxf(v[4 * k4 + 3] + b.w, 0.f);
                    }
#pragma unroll
                    for (int ch = 0; ch < N_CLASS; ++ch) {
                        const float4* w4 = reinterpret_cast<const float4*>(c.fw + F_WS2 + ch * 128 + f0);
#pragma unroll
                        for (int k4 = 0; k4 < 8; ++k4) {
                            const float4 w = w4[k4];
                            sl[ch] = fmaf(w.x, v[4 * k4], sl[ch]); sl[ch] = fmaf(w.y, v[4 * k4 + 1], sl[ch]);
                            sl[ch] = fmaf(w.z, v[4 * k4 + 2], sl[ch]); sl[ch] = fmaf(w.w, v[4 * k4 + 3], sl[ch]);
                        }
                    }
                }
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) c.part[(3 + h * 5 + ch) * TC_LD + p] = sl[ch];
            }
            T3_MARK(55);
            umma::fence_before_sync();
            t3_cons_sync();
            if (h == 0) {
                const float* P = c.part;
                float zl[N_CLASS], rgb[3];
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) zl[ch] = c.fw[F_BS2 + ch] + (P[(3 + ch) * TC_LD + p] + P[(8 + ch) * TC_LD + p]);
#pragma unroll
                for (int ch = 0; ch < 3; ++ch) rgb[ch] = SDF_ONLY ? 0.f : c.fw[F_BR + ch] + (rgb_e[ch] + P[ch * TC_LD + p]);
                float mx = zl[0];
#pragma unroll
                for (int ch = 1; ch < N_CLASS; ++ch) mx = fmaxf(mx, zl[ch]);
                float pr[N_CLASS], se = 0.f;
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) { pr[ch] = expf(zl[ch] - mx); se += pr[ch]; }
                float ent = 0.f, ex = 0.f;
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) {
                    pr[ch] = pr[ch] / se;
                    ent += pr[ch] * log2f(pr[ch] + 1e-5f);
                    ex += pr[ch] * (float)ch;
                }
                float* O = c.out;
                O[0 * TC_LD + p] = rgb[0]; O[1 * TC_LD + p] = rgb[1]; O[2 * TC_LD + p] = rgb[2];
                O[3 * TC_LD + p] = (ex / 4.0f - 0.5f) * 2.0f;
                O[4 * TC_LD + p] = -1.0f * ent;
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) O[(5 + ch) * TC_LD + p] = pr[ch];
            }
            t3_cons_sync();
            T3_MARK(56);
            epi.store(c.out, TC_LD, TC_TP, tile, N, c.tid, T3_GT);
            t3_cons_sync();
            T3_MARK(57);
        }
        ok = c.ok;
    }
    if (!ok && err) atomicExch(err, 1);
    mf_pdl_trigger();                                    // every tile of this CTA is drawn: the next kernel may start its prologue
    umma::fence_before_sync();
    __syncthreads();
    if (prof && blockIdx.x == 0 && threadIdx.x == 0) prof[28] = clock64();
    if (prof && threadIdx.x == 0 && blockIdx.x < 256) prof[65 + 2 * blockIdx.x] = mf_globaltimer();
    if (tile_ctr && threadIdx.x == 0 && atomicAdd(tile_ctr + 1, 1) == (int)gridDim.x - 1) {     // last CTA out re-arms the counter pair
        tile_ctr[0] = 0; tile_ctr[1] = 0;
        __threadfence();
    }
    if ((threadIdx.x >> 5) == 0) umma::tmem_dealloc<512>(tmem);
}
