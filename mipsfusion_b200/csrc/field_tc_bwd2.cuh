// Tensor-core (tcgen05) backward of the fused field evaluation, role-split version (the default; field_tc_bwd.cuh keeps
// the single-role kernel for A/B and for the pose-gradient route).  One persistent CTA per SM, 16 warps, 128 points per tile:
//
//   warps 4-11  CHAIN    the serial dependency chain of a tile: reload the encoded operand words (feature cache), forward
//                        layers 1-3, heads (softmax forward / backward), dZ3, dgrad3, dH, dgrad2, dZ1.  Two threads per point
//                        (64 features each).  After each layer's dZ is in tensor memory (and its dgrad is issued) the two
//                        warps that own a 32-point quarter copy the operands of that quarter's wgrad products -- bf16 hi / lo
//                        [point][feature] rows -- into one of two staging buffers in shared memory (quarter q uses buffer
//                        q & 1: quarters 0 / 1 and 2 / 3 fill in parallel, a buffer is refilled while the MMAs of the other one
//                        run) and issue the quarter's MMAs themselves (both operands MN-major from shared memory, bf16x3):
//                          dW[n][k] += sum_p dZ[p][n] X[p][k]                       (the three 128-wide layers)
//                          dV[n][c] += sum_p A[p][n] U[p][c],  U = [dlogits 5 | dRGB 3 | 0..]   (the two narrow heads:
//                             A = H3 gives sdf_linear.2.weight; A = [e | rgb_emb] gives rgb_linear.0.weight; the ones
//                             column of e gives both head biases) -- no warp-shuffle reductions over points anywhere.
//   warps 12-15 WGRAD    after the last quarter of a layer reads the 128 x K result from tensor memory and adds it to the CTA's
//                        partial gradient (coalesced reductions; every element has one owner thread).
//   warps 0-3   SCATTER  one thread per point: takes d(grid features) of the tile straight from the dgrad3 accumulator and
//                        scatters it into the hash-table gradient (128 reductions per point; the reduction rate of the SM is
//                        the bound of this stage, it no longer blocks the warps that feed the tensor core).
// (role order by warp id: the scheduler prefers the highest eligible warp id; the reductions are throughput work.)
//
// WGRAD's read-out and SCATTER's reductions of tile k run while the chain is already in tile k+1.  Hand-offs are mbarriers
// only (free / iss per staged quarter, dw_ready / dw_free per layer, dg3 / dcons around the accumulator columns SCATTER reads,
// w1 for the TMA copy below).
//
// Shared memory: W2 | W3 images resident (128 KB) | two 32 KB staging buffers | fp32 section | logit partials.  The W1 image
// (32 KB) lives in staging buffer 0 only while it is needed (forward layer 1): a TMA bulk copy (cp.async.bulk, async proxy)
// brings it in at the start of every tile, after the last wgrad MMAs that read the buffer have completed.
//
// Bias gradients cost nothing per point: pts_linear.0.bias and sdf_linear.0.bias are a ones column appended to the wgrad X
// operand (layer-1 slot 15, layer-3 feature 96), pts_linear.2.bias is linear in the other gradients
// (db2[:64] = Ws1[:, :64]^T dbs1, db2[64:] = Wr[:, :64]^T dbr) and is formed after the reduction over CTAs.
//
// Tensor memory: D [0,128) chain accumulator | R1 [128,256) e, H1, dZ3, dZ1 (hi, lo) | R2 [256,384) x3 = [sdf_emb | grid],
//                dH (hi, lo) | DW [384,512) wgrad accumulator.
// Activations that a later wgrad needs but tensor memory has no room for (H1, H3, rgb_emb: bf16 hi / lo words) are parked in
// a CTA-private scratch in global memory (L2 resident, [word][point]).
//
// Measured on B200 at C1 (98.7 k active of 176 k points; scripts/prof_bwd2.py): 0.265 ms vs 0.300 ms for the single-role
// kernel.  What the time is: the chain's own work is ~40 k cycles per tile, the five staged products add ~30 k (per product:
// stores 0.7 k, fence + quarter barrier + issue 1-1.8 k, MMA -> free 0.9 k, twice), and every load / store unit operation of
// the chain queues behind SCATTER's reductions (without them the kernel takes 0.24 ms).
#pragma once
#include "field_tc_bwd.cuh"

namespace b2 {

constexpr int B2_NT = 512, CHAIN_NT = 256, WG_NT = 128, SC_NT = 128;
constexpr int QROWS = 32;                              // points per staged quarter tile
constexpr uint32_t QBLK = QROWS * 128;                 // one 64-feature block of a quarter tile (4 KB)
// ---- shared memory map ----
constexpr int S_W = 0;                                 // weight image bytes [IMG_W2_HI, IMG_F32): W2 | W3, each hi then lo (128 KB)
constexpr int W2H = 0, W2L = IMG_W2_LO - IMG_W2_HI, W3H = IMG_W3_HI - IMG_W2_HI, W3L = IMG_W3_LO - IMG_W2_HI;
constexpr int S_ST = IMG_F32 - IMG_W2_HI;              // two staging buffers of 32 KB: A tile (hi 2 blocks, lo 2 blocks) | B tile
constexpr int ST_A = 0, ST_B = 4 * (int)QBLK, ST_BYTES = 8 * (int)QBLK;
constexpr int W1H = S_ST + IMG_W1_HI, W1L = S_ST + IMG_W1_LO;   // buffer 0 holds the W1 image during the forward layers (TMA, per tile)
constexpr int S_F32 = S_ST + 2 * ST_BYTES;             // fp32 section of the image
constexpr int S_PART = S_F32 + ((F_COUNT * 4 + 127) / 128) * 128;
constexpr int PART_ROWS = 10;                          // logit partial sums: 2 halves x 5 classes
constexpr int S_BAR = S_PART + PART_ROWS * TC_LD * 4;
constexpr int S_BYTES = S_BAR + 256;
constexpr size_t SMEM = S_BYTES + 1024;
static_assert(SMEM <= 227 * 1024, "shared memory budget");
// ---- tensor memory map ----
constexpr int T_D = 0, T_R1_HI = 128, T_R1_LO = 192, T_R2_HI = 256, T_R2_LO = 320, T_DW = 384;
constexpr int T_G_HI = T_R2_HI + 32, T_G_LO = T_R2_LO + 32;
// ---- CTA-private scratch in global memory, uint32 [word][point] ----
constexpr int SCR_H1 = 0, SCR_H3 = 128, SCR_RGB = 256, SCR_U = 320, SCR_WORDS = 328;     // hi words first, then lo words, per region (U: four-role kernel only)
constexpr int64_t SCR_CTA_WORDS = (int64_t)SCR_WORDS * TC_TP;
constexpr int REGS_CHAIN = 160, REGS_WGRAD = 88, REGS_SCATTER = 104;       // 256 x 160 + 128 x 88 + 128 x 104 = 65,536
// ---- mbarriers ----
enum { B_MMA = 0, B_DG3, B_DCONS, B_DWFREE, B_DWRDY, B_W1, B_IMG, B_FREE0, B_ISS0 = B_FREE0 + 4, B_COUNT = B_ISS0 + 4 };   // B_FREE0 + q: MMAs of staged quarter q done
constexpr int N_X3 = 112;                              // wgrad-3 X width: 64 sdf_emb + 32 grid + ones column + padding to 16

__device__ __forceinline__ void chain_sync() { asm volatile("bar.sync 1, %0;" ::"n"(CHAIN_NT) : "memory"); }
__device__ __forceinline__ void wg_sync() { asm volatile("bar.sync 2, %0;" ::"n"(WG_NT) : "memory"); }

struct Ctx {
    uint8_t* base; const float* fw; float* part; uint64_t* bars;
    uint32_t tmem, lane_base;
    bool ok;
};

// ---- MMA issue helpers (one thread).  Fully unrolled with the shared-memory descriptors formed by adding constants to one base
// descriptor (the start-address field counts 16-byte units): ~4 instructions per MMA instead of ~40 in a rolled loop that
// rebuilds the descriptor -- the other 255 threads of the chain wait while this thread issues. ----
// forward layer: D = A W^T, A at TMEM columns a_col(ks, lo), W image K-major at byte offsets (w_hi_off, w_lo_off)
template <int KS, class ColFn>
__device__ __forceinline__ void issue_fwd(const Ctx& c, int w_hi_off, int w_lo_off, ColFn a_col) {
    constexpr uint32_t idesc = umma::idesc_bf16(128, 128, 0, 0);
    const uint64_t dh = umma::smem_desc_sw128(umma::smem_u32(c.base + S_W + w_hi_off), 16, 1024);
    const uint64_t dl = umma::smem_desc_sw128(umma::smem_u32(c.base + S_W + w_lo_off), 16, 1024);
#pragma unroll
    for (int pass = 0; pass < 3; ++pass)
#pragma unroll
        for (int ks = 0; ks < KS; ++ks) {
            const uint32_t off = (uint32_t)(((ks >> 2) * IMG_BLOCK + (ks & 3) * 32) >> 4);
            umma::mma_ts(c.tmem + T_D, c.tmem + (uint32_t)a_col(ks, pass == 2), (pass == 1 ? dl : dh) + off, idesc, (pass | ks) ? 1u : 0u);
        }
}
// D[p][k] = sum_n dZ[p][n] W[n][k]: dZ (128 features, hi / lo) in region a_hi / a_lo, W image read MN-major, N_OUT columns
template <int N_OUT>
__device__ __forceinline__ void issue_dgrad(const Ctx& c, int a_hi, int a_lo, int w_hi_off, int w_lo_off) {
    constexpr uint32_t idesc = umma::idesc_bf16(128, N_OUT, 0, 1);
    const uint64_t dh = umma::smem_desc_sw128(umma::smem_u32(c.base + S_W + w_hi_off), IMG_BLOCK, 1024);
    const uint64_t dl = umma::smem_desc_sw128(umma::smem_u32(c.base + S_W + w_lo_off), IMG_BLOCK, 1024);
#pragma unroll
    for (int pass = 0; pass < 3; ++pass)
#pragma unroll
        for (int ks = 0; ks < 8; ++ks)
            umma::mma_ts(c.tmem + T_D, c.tmem + (uint32_t)((pass == 2 ? a_lo : a_hi) + 8 * ks), (pass == 1 ? dl : dh) + (uint32_t)((ks * 2048) >> 4),
                         idesc, (pass | ks) ? 1u : 0u);
}

__device__ __forceinline__ void ld32f(uint32_t taddr, float (&v)[32]) {
    uint32_t r[32];
    umma::tmem_ld32(taddr, r);
    umma::wait_ld();
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// store 32 packed words (hi 16, lo 16) of features [f0, f0+32) of this thread's point into an operand region
__device__ __forceinline__ void st_op(const Ctx& c, int hi_col, int lo_col, int f0, const uint32_t (&hi)[16], const uint32_t (&lo)[16]) {
    umma::tmem_st16(c.lane_base + (uint32_t)(hi_col + f0 / 2), hi);
    umma::tmem_st16(c.lane_base + (uint32_t)(lo_col + f0 / 2), lo);
}
__device__ __forceinline__ void split32(const float (&v)[32], uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
    for (int i = 0; i < 16; ++i) umma::split2(v[2 * i], v[2 * i + 1], hi[i], lo[i]);
}

// Staging stores with everything that depends on the thread folded into 8 precomputed shared-memory addresses:
// P[j] = address of 16-byte chunk j of this thread's row in its 64-feature block (block h of a tile at offset 0, 128-byte
// swizzle: chunk j sits at (j ^ (row & 7)) * 16); the tile and lo-part offsets are immediates -> one instruction per store.
template <int OFF>
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c_, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0+%1], {%2, %3, %4, %5};" ::"r"(addr), "n"(OFF), "r"(a), "r"(b), "r"(c_), "r"(d) : "memory");
}
template <int TILE_OFF, int CC>                         // 32 features = half CC of the block: chunks 4 CC .. 4 CC + 3
__device__ __forceinline__ void put32(const uint32_t (&P)[8], const uint32_t (&pk)[16]) {
#pragma unroll
    for (int c_ = 0; c_ < 4; ++c_) sts128<TILE_OFF>(P[4 * CC + c_], pk[4 * c_], pk[4 * c_ + 1], pk[4 * c_ + 2], pk[4 * c_ + 3]);
}
template <int TILE_OFF, int SG>                         // 16 features = slot group SG of the block: chunks 2 SG, 2 SG + 1
__device__ __forceinline__ void put16(const uint32_t (&P)[8], const uint32_t (&pk)[8]) {
#pragma unroll
    for (int c_ = 0; c_ < 2; ++c_) sts128<TILE_OFF>(P[2 * SG + c_], pk[4 * c_], pk[4 * c_ + 1], pk[4 * c_ + 2], pk[4 * c_ + 3]);
}
template <int TILE_OFF>                                 // this thread's 64 features of a tile: hi words and lo words (2 blocks later)
__device__ __forceinline__ void put64(const uint32_t (&P)[8], const uint32_t (&wh)[2][16], const uint32_t (&wl)[2][16]) {
    put32<TILE_OFF, 0>(P, wh[0]); put32<TILE_OFF, 1>(P, wh[1]);
    put32<TILE_OFF + 2 * (int)QBLK, 0>(P, wl[0]); put32<TILE_OFF + 2 * (int)QBLK, 1>(P, wl[1]);
}

// park / reload 32 packed words (hi 16 at word w0.., lo 16 at word 64 + w0.. of a 128-word region; 32 + w0.. for the 64-word
// rgb_emb region) of this thread's point in the CTA scratch; L2 only (the same thread re-reads what it wrote)
__device__ __forceinline__ void scr_store(uint32_t* scr_p, int region, int lo_off, int w0, const uint32_t (&hi)[16], const uint32_t (&lo)[16]) {
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        __stcg(scr_p + (size_t)(region + w0 + t) * TC_TP, hi[t]);
        __stcg(scr_p + (size_t)(region + lo_off + w0 + t) * TC_TP, lo[t]);
    }
}
__device__ __forceinline__ void scr_load(const uint32_t* scr_p, int region, int lo_off, int w0, uint32_t (&hi)[16], uint32_t (&lo)[16]) {
#pragma unroll
    for (int t = 0; t < 16; ++t) {
        hi[t] = __ldcg(scr_p + (size_t)(region + w0 + t) * TC_TP);
        lo[t] = __ldcg(scr_p + (size_t)(region + lo_off + w0 + t) * TC_TP);
    }
}

}  // namespace b2

// ---------------------------------------------------------------------------------------------
// The kernel (parameter gradients only; ray / point gradients use field_bwd_tc_kernel<Src, true>).
// part: [gridDim.x][MF_MLP_PARAMS] per-CTA partial parameter gradients (zeroed here);
// scratch: [gridDim.x][SCR_CTA_WORDS] uint32.
// ---------------------------------------------------------------------------------------------
template <class Src>
__global__ void __launch_bounds__(b2::B2_NT, 1) field_bwd_tc2_kernel(FieldDev f, Src src, const float* __restrict__ d_raw,
                                                                  float* __restrict__ grad_grid, float* __restrict__ part,
                                                                  uint32_t* __restrict__ scratch, int64_t N_all, ActiveMap am,
                                                                  int* __restrict__ err, long long* __restrict__ prof, int agg) {
    using namespace b2;
    extern __shared__ uint8_t smem_raw[];
    const int tid = threadIdx.x, warp = tid >> 5;
    mf_pdl_wait();                                       // (programmatic launch, mf_common.cuh: no global access before it)
    if (prof && tid == 0 && blockIdx.x < 256) prof[576 + 2 * blockIdx.x] = mf_globaltimer();
    float* gpart = part + (size_t)blockIdx.x * MF_MLP_PARAMS;
    for (int i = tid; i < MF_MLP_PARAMS; i += B2_NT) gpart[i] = 0.f;

    Ctx c;
    c.base = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
    c.fw = (const float*)(c.base + S_F32); c.part = (float*)(c.base + S_PART); c.bars = (uint64_t*)(c.base + S_BAR);
    uint32_t* tmem_ptr = (uint32_t*)(c.base + S_BAR + 8 * B_COUNT);
    if (warp == 0) umma::tmem_alloc<512>(tmem_ptr);
    if (tid == 0) {
        umma::mbar_init(c.bars + B_MMA, 1); umma::mbar_init(c.bars + B_DG3, 1); umma::mbar_init(c.bars + B_DCONS, SC_NT);
        umma::mbar_init(c.bars + B_DWFREE, WG_NT); umma::mbar_init(c.bars + B_DWRDY, 4); umma::mbar_init(c.bars + B_W1, 1);
        umma::mbar_init(c.bars + B_IMG, 1);
        for (int q = 0; q < 4; ++q) { umma::mbar_init(c.bars + B_FREE0 + q, 1); umma::mbar_init(c.bars + B_ISS0 + q, 1); }
        umma::fence_barrier_init();
        // resident weights (W2 | W3 images, fp32 section) through the bulk-copy engine while the CTA zero-fills its partials
        constexpr uint32_t W_BYTES = IMG_F32 - IMG_W2_HI, F_BYTES = F_COUNT * 4, CHUNK = 32768;
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(umma::smem_u32(c.bars + B_IMG)), "r"(W_BYTES + F_BYTES) : "memory");
        for (uint32_t off = 0; off < W_BYTES; off += CHUNK)
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(umma::smem_u32(c.base + S_W + off)), "l"(f.tc_img + IMG_W2_HI + off), "r"(W_BYTES - off < CHUNK ? W_BYTES - off : CHUNK),
                           "r"(umma::smem_u32(c.bars + B_IMG)) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                     ::"r"(umma::smem_u32(c.base + S_F32)), "l"(f.tc_img + IMG_F32), "r"(F_BYTES), "r"(umma::smem_u32(c.bars + B_IMG)) : "memory");
    }
    umma::fence_before_sync();
    __syncthreads();                                   // also orders the gpart zero-fill before WGRAD's reductions
    umma::fence_after_sync();
    c.tmem = *tmem_ptr;
    c.lane_base = c.tmem + ((uint32_t)((warp & 3) * 32) << 16);
    c.ok = umma::mbar_wait(c.bars + B_IMG, 0);         // the weights have landed

    const int64_t N = am.n(N_all);                     // active points only (ascending point indices in am.idx)
    const int64_t n_tiles = (N + TC_TP - 1) / TC_TP;
    const int p = tid & (TC_TP - 1);
#define B2_MARK(slot) do { if (prof && blockIdx.x == 0 && k == 1 && (ctid & 127) == 0) prof[slot] = clock64(); } while (0)

    // Role order SCATTER (warps 0-3), CHAIN (4-11), WGRAD (12-15): the warp scheduler prefers the highest eligible warp id.
    // The MMA issuer must react at once to a staged quarter (measured: 1.4-1.8 k cycles late when it sat below the chain's
    // warps), the chain's instructions are latency critical, the reductions of SCATTER are throughput work.
    const int ctid = tid - SC_NT;                      // thread index inside the chain (outside [0, 256) for the other roles)
    if (ctid >= 0 && ctid < CHAIN_NT) {
        // =============================== CHAIN ===============================
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(REGS_CHAIN));
        const int h = ctid >> 7;
        uint32_t ph_mma = 0;
        uint32_t k = 0;
        auto round = [&](auto issue) {                 // publish TMEM stores, rendezvous, thread 0 issues + commits, all wait
            umma::wait_st();
            umma::fence_before_sync();
            chain_sync();
            if (ctid == 0) { umma::fence_after_sync(); issue(); umma::commit(c.bars + B_MMA); }
            c.ok &= umma::mbar_wait_spin(c.bars + B_MMA, ph_mma);
            ph_mma ^= 1;
            umma::fence_after_sync();
        };
        // ---- wgrad products: 5 per tile, each streamed in 4 quarters (the 32 points of a lane quadrant) through the staging
        // buffer quarter & 1.  prod = global product counter (5 k + P):
        //   P = 0  dWs1 (+ dbs1) = dZ3^T [sdf_emb | grid | 1]    -> DW[0, 112)      P = 1  dWs2 = H3^T U              -> DW[112, 128)
        //   P = 2  dW2 = dH^T H1                                 -> DW[0, 128)
        //   P = 3  dW1 (+ db1) = dZ1^T e (ones in slot 15)       -> DW[0, 64)       P = 4  [e | rgb_emb]^T U -> DW[64, 80)
        // A buffer is free once the MMAs of the quarter that used it before have completed (`free`, one completion per product
        // and quarter).  The two warps of a quarter write their rows, make them visible to the tensor core, and lane 0 of the
        // h = 0 warp issues the quarter's MMAs: passes (A hi, B hi), (A lo, B hi), (A hi, B lo) over two 16-point k-steps.  The
        // issue order q0 < q1 < q2 < q3 is enforced (`iss`): deterministic accumulation order, and q0's first MMA overwrites.
        const int row = p & (QROWS - 1), quarter = p >> 5, lane = tid & 31;
        uint32_t PA[8], PH[8], PQ[4];                  // chunk addresses of this thread's row: block 0 / block h / its half of block 0
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            PA[j] = umma::smem_u32(c.base) + (uint32_t)(S_ST + (quarter & 1) * ST_BYTES) + (uint32_t)((row >> 3) * 1024 + (row & 7) * 128) +
                    (uint32_t)(((j ^ row) & 7) << 4);
            PH[j] = PA[j] + (uint32_t)h * QBLK;
        }
#pragma unroll
        for (int c_ = 0; c_ < 4; ++c_) PQ[c_] = h ? PA[4 + c_] : PA[c_];
        const uint64_t dA0 = umma::desc_mn(c.base + S_ST + (quarter & 1) * ST_BYTES + ST_A, 0, QBLK);
        const uint64_t dB0 = umma::desc_mn(c.base + S_ST + (quarter & 1) * ST_BYTES + ST_B, 0, QBLK);
        constexpr uint32_t LO_STEP = (2 * QBLK) >> 4, KS_STEP = (16 * 128) >> 4;
        auto prod_begin = [&](uint32_t prod) {
            c.ok &= umma::mbar_wait_spin(c.bars + B_FREE0 + ((quarter + 2) & 3), quarter >= 2 ? (prod & 1u) : ((prod + 1u) & 1u));
        };
        auto prod_end = [&](int PK, uint32_t prod, uint32_t lay) {
            umma::fence_proxy_async();
            asm volatile("bar.sync %0, 64;" ::"r"(3 + quarter) : "memory");
            if (h == 0 && lane == 0) {
                umma::fence_after_sync();
                if (quarter == 0) {
                    if (PK == 0 || PK == 2 || PK == 3) c.ok &= umma::mbar_wait_spin(c.bars + B_DWFREE, (lay + 1u) & 1u);   // previous layer read out
                } else {
                    c.ok &= umma::mbar_wait_spin(c.bars + B_ISS0 + quarter - 1, prod & 1u);
                }
                const int n_out = PK == 0 ? N_X3 : (PK == 2 ? D_H : (PK == 3 ? 64 : 16));
                const uint32_t idesc = umma::idesc_bf16(128, n_out, 1, 1);
                const uint32_t dcol = c.tmem + (uint32_t)(T_DW + (PK == 1 ? N_X3 : (PK == 4 ? 64 : 0)));
#pragma unroll
                for (int j = 0; j < 6; ++j) {
                    const int pass = j >> 1, ks = j & 1;
                    umma::mma_ss(dcol, dA0 + (uint64_t)((pass == 1 ? LO_STEP : 0) + ks * KS_STEP),
                                 dB0 + (uint64_t)((pass == 2 ? LO_STEP : 0) + ks * KS_STEP), idesc, (j == 0 && quarter == 0) ? 0u : 1u);
                }
                umma::mbar_arrive(c.bars + B_ISS0 + quarter);
                umma::commit(c.bars + B_FREE0 + quarter);
                if (PK == 1 || PK == 2 || PK == 4) umma::commit(c.bars + B_DWRDY);       // (covers this thread's MMAs of P - 1 too)
            }
        };
        // U = [dlogits 5 | dRGB 3 | 0 x 8] -> features 0 .. 15 of the B tile; the h = 0 thread writes the hi part, h = 1 the lo part
        auto put_u = [&](const uint32_t (&uh)[4], const uint32_t (&ul)[4]) {
            if (h == 0) { sts128<ST_B>(PA[0], uh[0], uh[1], uh[2], uh[3]); sts128<ST_B>(PA[1], 0u, 0u, 0u, 0u); }
            else { sts128<ST_B + 2 * (int)QBLK>(PA[0], ul[0], ul[1], ul[2], ul[3]); sts128<ST_B + 2 * (int)QBLK>(PA[1], 0u, 0u, 0u, 0u); }
        };
        // W1 image -> staging buffer 0 by the TMA (async proxy: no thread copies anything); issued by one thread
        auto load_w1 = [&]() {
            umma::fence_proxy_async();
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(umma::smem_u32(c.bars + B_W1)), "r"(2 * IMG_BLOCK) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(umma::smem_u32(c.base + S_ST)), "l"(f.tc_img + IMG_W1_HI), "r"(2 * IMG_BLOCK), "r"(umma::smem_u32(c.bars + B_W1))
                         : "memory");
        };
        uint32_t* scr_p = scratch + (size_t)blockIdx.x * SCR_CTA_WORDS + p;
        // copy this thread's 64 dZ features (two 32-feature groups) from an operand region into the Z staging tile
        // this thread's 64 dZ features (two 32-feature groups) of an operand region: load (one TMEM round trip) / store to ZS
        auto load_z = [&](int r_hi, int r_lo, uint32_t (&wh)[2][16], uint32_t (&wl)[2][16]) {
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                umma::tmem_ld16(c.lane_base + (uint32_t)(r_hi + 16 * (2 * h + cc)), wh[cc]);
                umma::tmem_ld16(c.lane_base + (uint32_t)(r_lo + 16 * (2 * h + cc)), wl[cc]);
            }
            umma::wait_ld();
        };

        int64_t i_next = 0;
        { const int64_t s0 = (int64_t)blockIdx.x * TC_TP + p; if (s0 < N) i_next = am(s0); }
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
            const int64_t slot = tile * TC_TP + p;
            const bool valid = slot < N;
            const int64_t i = i_next;                                       // (loaded one tile ahead)
            { const int64_t s1 = slot + (int64_t)gridDim.x * TC_TP; i_next = s1 < N ? am(s1) : 0; }
            // (prefetching the next tile's cached operand words into L2 here shortened the load phase by 2 k cycles but cost more in
            // load / store unit traffic than it saved: 0.287 vs 0.273 ms)
            const uint32_t lay0 = 3u * k, prod0 = 5u * k;                   // global layer / product counters of this tile
            if (ctid == 0) {                                                // W1 -> staging buffer 0 (last used by quarters 0 and 2 of product 4)
                if (k > 0) {
                    c.ok &= umma::mbar_wait_spin(c.bars + B_FREE0 + 0, (prod0 - 1u) & 1u);
                    c.ok &= umma::mbar_wait_spin(c.bars + B_FREE0 + 2, (prod0 - 1u) & 1u);
                }
                load_w1();
            }
            B2_MARK(0);
            float g[3], gs[7];                                 // d loss / d (rgb 3 | sdf, entropy, prob[5])
            {
                const float2* gr = reinterpret_cast<const float2*>(d_raw + i * MF_RAW_DIM);       // 40-byte rows: 8-byte aligned
                float2 t2[5];
#pragma unroll
                for (int j = 0; j < 5; ++j) t2[j] = valid ? __ldg(gr + j) : make_float2(0.f, 0.f);
                g[0] = t2[0].x; g[1] = t2[0].y; g[2] = t2[1].x;
                gs[0] = t2[1].y; gs[1] = t2[2].x; gs[2] = t2[2].y; gs[3] = t2[3].x; gs[4] = t2[3].y; gs[5] = t2[4].x; gs[6] = t2[4].y;
            }
            float x[3] = {0.f, 0.f, 0.f};
            if (!f.feat && valid) src.point(i, f, x);
            // operand words the forward kernel cached: [i / 128][slot group 4][word 24][i % 128]
            const uint32_t* fin = f.feat ? f.feat + (size_t)(i >> 7) * FEAT_TILE_WORDS + (i & (TC_TP - 1)) : nullptr;
            // the 8 hi + 8 lo words of slot group qq of this thread's point (cached by the forward, or recomputed)
            auto e_words = [&](int qq, uint32_t (&hi)[8], uint32_t (&lo)[8]) {
                if (fin) {
                    const uint32_t* fq = fin + (size_t)qq * FEAT_WORDS * TC_TP;
#pragma unroll
                    for (int t = 0; t < 8; ++t) { hi[t] = __ldg(fq + t * TC_TP); lo[t] = __ldg(fq + (8 + t) * TC_TP); }
                } else {
                    float e[16];
                    tb_e_slots(x, qq, e);
#pragma unroll
                    for (int t = 0; t < 8; ++t) umma::split2(e[2 * t], e[2 * t + 1], hi[t], lo[t]);
                }
            };
            // ---- layer-1 operand e (slot groups 2h, 2h+1) -> R1, grid features (levels 8h .. 8h+7) -> R2 ----
#pragma unroll
            for (int sg = 0; sg < 2; ++sg) {
                const int qq = 2 * h + sg;
                uint32_t hi[8], lo[8], gh[4], gl[4];
                e_words(qq, hi, lo);
                if (fin) {
                    const uint32_t* fq = fin + (size_t)qq * FEAT_WORDS * TC_TP;
#pragma unroll
                    for (int t = 0; t < 4; ++t) { gh[t] = __ldg(fq + (16 + t) * TC_TP); gl[t] = __ldg(fq + (20 + t) * TC_TP); }
                } else {
                    float gf[8];
                    const float2* grid2 = reinterpret_cast<const float2*>(f.grid);
#pragma unroll
                    for (int ll = 0; ll < 4; ++ll) {
                        float2 vv = make_float2(0.f, 0.f);
                        if (valid) vv = grid_level_fwd(x, grid2, level_info(f, qq * 4 + ll), nullptr);
                        gf[2 * ll] = vv.x; gf[2 * ll + 1] = vv.y;
                    }
#pragma unroll
                    for (int t = 0; t < 4; ++t) umma::split2(gf[2 * t], gf[2 * t + 1], gh[t], gl[t]);
                }
                umma::tmem_st8(c.lane_base + T_R1_HI + 8 * qq, hi);
                umma::tmem_st8(c.lane_base + T_R1_LO + 8 * qq, lo);
                umma::tmem_st4(c.lane_base + T_G_HI + 4 * qq, gh);
                umma::tmem_st4(c.lane_base + T_G_LO + 4 * qq, gl);
            }
            B2_MARK(1);
            float v[32];
            uint32_t mask1[2], mask3[2];
            // ---- forward layer 1 ----
            round([&]() {
                c.ok &= umma::mbar_wait_spin(c.bars + B_W1, k & 1u);           // the W1 image has landed in staging buffer 0
                issue_fwd<4>(c, W1H, W1L, [](int ks, bool lo) { return (lo ? T_R1_LO : T_R1_HI) + 8 * ks; });
            });
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
                const int f0 = 64 * h + 32 * cc;
                ld32f(c.lane_base + T_D + f0, v);
                const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_B1 + f0);
                uint32_t m = 0;
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 b = b4[k4];
                    v[4 * k4] = fmaxf(v[4 * k4] + b.x, 0.f); v[4 * k4 + 1] = fmaxf(v[4 * k4 + 1] + b.y, 0.f);
                    v[4 * k4 + 2] = fmaxf(v[4 * k4 + 2] + b.z, 0.f); v[4 * k4 + 3] = fmaxf(v[4 * k4 + 3] + b.w, 0.f);
                }
#pragma unroll
                for (int kk = 0; kk < 32; ++kk) m |= (v[kk] > 0.f ? 1u : 0u) << kk;
                mask1[cc] = m;
                uint32_t hi[16], lo[16];
                split32(v, hi, lo);
                st_op(c, T_R1_HI, T_R1_LO, f0, hi, lo);                      // H1: A operand of layer 2 ...
                scr_store(scr_p, SCR_H1, 64, f0 / 2, hi, lo);                // ... and, parked, the X operand of its wgrad
            }
            B2_MARK(2);
            // ---- forward layer 2 ----
            round([&]() { issue_fwd<8>(c, W2H, W2L, [](int ks, bool lo) { return (lo ? T_R1_LO : T_R1_HI) + 8 * ks; }); });
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
                const int f0 = 64 * h + 32 * cc;
                ld32f(c.lane_base + T_D + f0, v);
                const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_B2 + f0);
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 b = b4[k4];
                    v[4 * k4] += b.x; v[4 * k4 + 1] += b.y; v[4 * k4 + 2] += b.z; v[4 * k4 + 3] += b.w;
                }
                uint32_t hi[16], lo[16];
                split32(v, hi, lo);
                if (h == 0) st_op(c, T_R2_HI, T_R2_LO, f0, hi, lo);          // sdf_emb -> layer-3 operand, features [0, 64)
                else scr_store(scr_p, SCR_RGB, 32, 16 * cc, hi, lo);         // rgb_emb: A operand of the colour-head wgrad
            }
            B2_MARK(3);
            // ---- forward layer 3 ----
            round([&]() {
                issue_fwd<6>(c, W3H, W3L, [](int ks, bool lo) {
                    return ks < 4 ? (lo ? T_R2_LO : T_R2_HI) + 8 * ks : (lo ? T_G_LO : T_G_HI) + 8 * (ks - 4);
                });
            });
            {
                float s[N_CLASS] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll 1
                for (int cc = 0; cc < 2; ++cc) {
                    const int f0 = 64 * h + 32 * cc;
                    ld32f(c.lane_base + T_D + f0, v);
                    const float4* b4 = reinterpret_cast<const float4*>(c.fw + F_BS1 + f0);
                    uint32_t m = 0;
#pragma unroll
                    for (int k4 = 0; k4 < 8; ++k4) {
                        const float4 b = b4[k4];
                        v[4 * k4] = fmaxf(v[4 * k4] + b.x, 0.f); v[4 * k4 + 1] = fmaxf(v[4 * k4 + 1] + b.y, 0.f);
                        v[4 * k4 + 2] = fmaxf(v[4 * k4 + 2] + b.z, 0.f); v[4 * k4 + 3] = fmaxf(v[4 * k4 + 3] + b.w, 0.f);
                    }
#pragma unroll
                    for (int kk = 0; kk < 32; ++kk) m |= (v[kk] > 0.f ? 1u : 0u) << kk;
                    mask3[cc] = m;
#pragma unroll
                    for (int ch = 0; ch < N_CLASS; ++ch) {
                        const float4* w4 = reinterpret_cast<const float4*>(c.fw + F_WS2 + ch * 128 + f0);
#pragma unroll
                        for (int k4 = 0; k4 < 8; ++k4) {
                            const float4 w = w4[k4];
                            s[ch] = fmaf(w.x, v[4 * k4], s[ch]); s[ch] = fmaf(w.y, v[4 * k4 + 1], s[ch]);
                            s[ch] = fmaf(w.z, v[4 * k4 + 2], s[ch]); s[ch] = fmaf(w.w, v[4 * k4 + 3], s[ch]);
                        }
                    }
                    uint32_t hi[16], lo[16];
                    split32(v, hi, lo);
                    scr_store(scr_p, SCR_H3, 64, f0 / 2, hi, lo);            // H3: A operand of the sdf_linear.2 wgrad
                }
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) c.part[(h * 5 + ch) * TC_LD + p] = s[ch];
            }
            B2_MARK(4);
            chain_sync();
            // ---- heads: softmax forward + backward (both threads of a point, redundantly) ----
            float dz4[N_CLASS];
            {
                float zl[N_CLASS], pr[N_CLASS], dp[N_CLASS];
                float mx = -INFINITY, se = 0.f, dot = 0.f;
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) {
                    zl[ch] = c.fw[F_BS2 + ch] + (c.part[ch * TC_LD + p] + c.part[(5 + ch) * TC_LD + p]);
                    mx = fmaxf(mx, zl[ch]);
                }
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) { pr[ch] = expf(zl[ch] - mx); se += pr[ch]; }
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) {
                    pr[ch] = pr[ch] / se;
                    const float qq = pr[ch] + 1e-5f;
                    dp[ch] = gs[2 + ch] + gs[0] * (0.5f * (float)ch) - gs[1] * (log2f(qq) + pr[ch] / (qq * 0.6931471805599453f));
                    dot = fmaf(pr[ch], dp[ch], dot);
                }
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) dz4[ch] = pr[ch] * (dp[ch] - dot);
            }
            // U = [dlogits 5 | dRGB 3 | 0 x 8] as bf16 hi / lo words (B operand of the two narrow-head wgrads)
            uint32_t uh[4], ul[4];
            umma::split2(dz4[0], dz4[1], uh[0], ul[0]); umma::split2(dz4[2], dz4[3], uh[1], ul[1]);
            umma::split2(dz4[4], g[0], uh[2], ul[2]); umma::split2(g[1], g[2], uh[3], ul[3]);
            // ---- dZ3 = (Ws2^T dz4) * relu'(h3) -> R1 (H1 is parked; its columns are free since the layer-2 MMAs completed) ----
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
                const int f0 = 64 * h + 32 * cc;
#pragma unroll
                for (int kk = 0; kk < 32; ++kk) v[kk] = 0.f;
#pragma unroll
                for (int ch = 0; ch < N_CLASS; ++ch) {
                    const float4* w4 = reinterpret_cast<const float4*>(c.fw + F_WS2 + ch * 128 + f0);
                    const float dzc = dz4[ch];
#pragma unroll
                    for (int k4 = 0; k4 < 8; ++k4) {
                        const float4 w = w4[k4];
                        v[4 * k4] = fmaf(w.x, dzc, v[4 * k4]); v[4 * k4 + 1] = fmaf(w.y, dzc, v[4 * k4 + 1]);
                        v[4 * k4 + 2] = fmaf(w.z, dzc, v[4 * k4 + 2]); v[4 * k4 + 3] = fmaf(w.w, dzc, v[4 * k4 + 3]);
                    }
                }
                const uint32_t m = mask3[cc];
#pragma unroll
                for (int kk = 0; kk < 32; ++kk) v[kk] = ((m >> kk) & 1u) ? v[kk] : 0.f;
                uint32_t zh[16], zl[16];
                split32(v, zh, zl);
                st_op(c, T_R1_HI, T_R1_LO, f0, zh, zl);
            }
            B2_MARK(5);
            // ---- dgrad of layer 3 (its completion also releases SCATTER on the grid-feature columns of D) ----
            umma::wait_st();
            umma::fence_before_sync();
            chain_sync();
            if (ctid == 0) {
                umma::fence_after_sync();
                issue_dgrad<D_SDF_IN>(c, T_R1_HI, T_R1_LO, W3H, W3L);
                umma::commit(c.bars + B_DG3);
            }
            // ... meanwhile, the two products of layer 3.  P0: A = dZ3 (R1), B = [sdf_emb | grid | 1] (R2); everything is in registers
            // before the wait, the critical section is shared-memory stores only.
            {
                uint32_t zh[2][16], zl[2][16], xh[2][16], xl[2][16];
                load_z(T_R1_HI, T_R1_LO, zh, zl);
                if (h == 0) {
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) { umma::tmem_ld16(c.lane_base + T_R2_HI + 16 * cc, xh[cc]); umma::tmem_ld16(c.lane_base + T_R2_LO + 16 * cc, xl[cc]); }
                } else {
                    umma::tmem_ld16(c.lane_base + T_G_HI, xh[0]); umma::tmem_ld16(c.lane_base + T_G_LO, xl[0]);
#pragma unroll
                    for (int t = 0; t < 16; ++t) { xh[1][t] = 0u; xl[1][t] = 0u; }
                    xh[1][0] = 0x00003F80u;                                  // feature 96 = 1.0 (bf16): bias column of sdf_linear.0
                }
                umma::wait_ld();
                if (prof && blockIdx.x == 0 && k == 1 && lane == 0 && h == 0) prof[32 + 4 * quarter] = clock64();
                prod_begin(prod0);
                if (prof && blockIdx.x == 0 && k == 1 && lane == 0 && h == 0) prof[33 + 4 * quarter] = clock64();
                put64<ST_A>(PH, zh, zl);
                put64<ST_B>(PH, xh, xl);
                if (prof && blockIdx.x == 0 && k == 1 && lane == 0 && h == 0) prof[34 + 4 * quarter] = clock64();
                prod_end(0, prod0, lay0);
                if (prof && blockIdx.x == 0 && k == 1 && lane == 0 && h == 0) prof[35 + 4 * quarter] = clock64();
                // P1: A = H3 (parked), B = U
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) scr_load(scr_p, SCR_H3, 64, 32 * h + 16 * cc, zh[cc], zl[cc]);
                prod_begin(prod0 + 1u);
                put64<ST_A>(PH, zh, zl);
                put_u(uh, ul);
                prod_end(1, prod0 + 1u, lay0);
            }
            B2_MARK(6);
            c.ok &= umma::mbar_wait_spin(c.bars + B_DG3, k & 1u);
            umma::fence_after_sync();
            B2_MARK(7);
            // ---- dH = [d sdf_emb (dgrad of layer 3), d rgb_emb (colour head)] -> R2 (this thread's x3 words are staged) ----
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
                const int f0 = 64 * h + 32 * cc;
                if (h == 0) {
                    ld32f(c.lane_base + T_D + f0, v);
                } else {
                    const float* wr = c.fw + F_WR_EMB + 32 * cc;
#pragma unroll
                    for (int kk = 0; kk < 32; ++kk) v[kk] = fmaf(wr[128 + kk], g[2], fmaf(wr[64 + kk], g[1], wr[kk] * g[0]));
                }
                uint32_t zh[16], zl[16];
                split32(v, zh, zl);
                st_op(c, T_R2_HI, T_R2_LO, f0, zh, zl);
            }
            // ---- dgrad of layer 2 (D is overwritten: SCATTER must have taken its columns) ----
            umma::wait_st();
            umma::fence_before_sync();
            chain_sync();
            if (ctid == 0) {
                c.ok &= umma::mbar_wait_spin(c.bars + B_DCONS, k & 1u);
                umma::fence_after_sync();
                issue_dgrad<D_H>(c, T_R2_HI, T_R2_LO, W2H, W2L);
                umma::commit(c.bars + B_MMA);
            }
            B2_MARK(8);
            // ... meanwhile, P2: A = dH (R2), B = H1 (parked)
            {
                uint32_t ah[2][16], al[2][16], zh[2][16], zl[2][16];
#pragma unroll
                for (int cc = 0; cc < 2; ++cc) scr_load(scr_p, SCR_H1, 64, 32 * h + 16 * cc, ah[cc], al[cc]);
                load_z(T_R2_HI, T_R2_LO, zh, zl);
                prod_begin(prod0 + 2u);
                put64<ST_A>(PH, zh, zl);
                put64<ST_B>(PH, ah, al);
                prod_end(2, prod0 + 2u, lay0 + 1u);
            }
            c.ok &= umma::mbar_wait_spin(c.bars + B_MMA, ph_mma);
            ph_mma ^= 1;
            umma::fence_after_sync();
            B2_MARK(9);
            // ---- dZ1 = dgrad2 * relu'(h1) -> R1 (dZ3 is staged and its dgrad done) ----
#pragma unroll 1
            for (int cc = 0; cc < 2; ++cc) {
                const int f0 = 64 * h + 32 * cc;
                ld32f(c.lane_base + T_D + f0, v);
                const uint32_t m = mask1[cc];
#pragma unroll
                for (int kk = 0; kk < 32; ++kk) v[kk] = ((m >> kk) & 1u) ? v[kk] : 0.f;
                uint32_t zh[16], zl[16];
                split32(v, zh, zl);
                st_op(c, T_R1_HI, T_R1_LO, f0, zh, zl);
            }
            umma::wait_st();
            // ---- the two products of layer 1.  P3: A = dZ1 (R1), B = e (ones in slot 15: bias column);
            //      P4: A = [e | rgb_emb (parked)] (the ones row gives both head biases), B = U.  Thread h owns slot groups 2h, 2h+1 of
            //      e (its half of block 0) and half h of rgb_emb (block 1) ----
            {
                uint32_t zh[2][16], zl[2][16], eh[2][8], el[2][8], rh[16], rl[16];
                load_z(T_R1_HI, T_R1_LO, zh, zl);
                e_words(2 * h, eh[0], el[0]); e_words(2 * h + 1, eh[1], el[1]);
                if (h == 0) { eh[0][7] = (eh[0][7] & 0x0000ffffu) | 0x3F800000u; el[0][7] &= 0x0000ffffu; }   // slot 15 = 1.0
                scr_load(scr_p, SCR_RGB, 32, 16 * h, rh, rl);
                prod_begin(prod0 + 3u);
                put64<ST_A>(PH, zh, zl);
#pragma unroll
                for (int sg = 0; sg < 2; ++sg)
#pragma unroll
                    for (int c_ = 0; c_ < 2; ++c_) {
                        sts128<ST_B>(PQ[2 * sg + c_], eh[sg][4 * c_], eh[sg][4 * c_ + 1], eh[sg][4 * c_ + 2], eh[sg][4 * c_ + 3]);
                        sts128<ST_B + 2 * (int)QBLK>(PQ[2 * sg + c_], el[sg][4 * c_], el[sg][4 * c_ + 1], el[sg][4 * c_ + 2], el[sg][4 * c_ + 3]);
                    }
                prod_end(3, prod0 + 3u, lay0 + 2u);
                prod_begin(prod0 + 4u);
#pragma unroll
                for (int sg = 0; sg < 2; ++sg)
#pragma unroll
                    for (int c_ = 0; c_ < 2; ++c_) {
                        sts128<ST_A>(PQ[2 * sg + c_], eh[sg][4 * c_], eh[sg][4 * c_ + 1], eh[sg][4 * c_ + 2], eh[sg][4 * c_ + 3]);
                        sts128<ST_A + 2 * (int)QBLK>(PQ[2 * sg + c_], el[sg][4 * c_], el[sg][4 * c_ + 1], el[sg][4 * c_ + 2], el[sg][4 * c_ + 3]);
                    }
#pragma unroll
                for (int c_ = 0; c_ < 4; ++c_) {
                    sts128<ST_A + (int)QBLK>(PQ[c_], rh[4 * c_], rh[4 * c_ + 1], rh[4 * c_ + 2], rh[4 * c_ + 3]);
                    sts128<ST_A + 3 * (int)QBLK>(PQ[c_], rl[4 * c_], rl[4 * c_ + 1], rl[4 * c_ + 2], rl[4 * c_ + 3]);
                }
                put_u(uh, ul);
                prod_end(4, prod0 + 4u, lay0 + 2u);
            }
            B2_MARK(10);
            umma::fence_before_sync();
            chain_sync();          // every accumulator / operand read of this tile is done before the next tile's stores
        }
    } else if (ctid >= CHAIN_NT) {
        // =============================== WGRAD ===============================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_WGRAD));
        const int wt = ctid - CHAIN_NT;                // = accumulator lane n
        // destination of this lane's row of the colour-head product [e | rgb_emb]^T U inside rgb_linear.0.weight (or -1)
        const int kin = wt >= 64 ? wt - 64 : (tc_e_slot_to_index(wt) >= 0 ? 64 + tc_e_slot_to_index(wt) : -1);
        uint32_t k = 0, lay = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
#pragma unroll 1
            for (int L = 0; L < 3; ++L, ++lay) {
                c.ok &= umma::mbar_wait_spin(c.bars + B_DWRDY, lay & 1u);
                umma::fence_after_sync();
                if (prof && blockIdx.x == 0 && k == 1 && wt == 0) prof[16 + L] = clock64();
                // read-out: lane n owns DW[n][*]; every element has one owner thread: reductions without return
                const int n_cols = L == 0 ? 128 : (L == 1 ? D_H : 80);
#pragma unroll 1
                for (int c0 = 0; c0 < n_cols; c0 += 16) {
                    uint32_t r[16];
                    umma::tmem_ld16(c.lane_base + (uint32_t)(T_DW + c0), r);
                    umma::wait_ld();
                    if (L == 1 || (L == 0 && c0 < D_SDF_IN)) {             // dW2 / dWs1: column kc -> [kc][n]
                        float* dst = gpart + (L == 1 ? OFF_W2 : OFF_WS1) + c0 * D_H + wt;
#pragma unroll
                        for (int j = 0; j < 16; ++j) atomicAdd(dst + j * D_H, __uint_as_float(r[j]));
                    } else if (L == 0) {
                        if (c0 == D_SDF_IN) {                              // ones column: dbs1
                            atomicAdd(&gpart[OFF_BS1 + wt], __uint_as_float(r[0]));
                        } else {                                           // H3^T U: dWs2[c][n]
#pragma unroll
                            for (int j = 0; j < N_CLASS; ++j) atomicAdd(&gpart[OFF_WS2 + j * D_H + wt], __uint_as_float(r[j]));
                        }
                    } else if (c0 < 64) {                                  // dW1: slot kc -> e index (slot 15 = ones column: db1)
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const int ei = tc_e_slot_to_index(c0 + j);
                            if (ei >= 0) atomicAdd(&gpart[OFF_W1 + ei * D_H + wt], __uint_as_float(r[j]));
                            else if (c0 + j == 15) atomicAdd(&gpart[OFF_B1 + wt], __uint_as_float(r[j]));
                        }
                    } else if (wt == 15) {                                 // the ones row of [e | rgb_emb]: sums of U over the points
#pragma unroll
                        for (int j = 0; j < N_CLASS; ++j) atomicAdd(&gpart[OFF_BS2 + j], __uint_as_float(r[j]));
#pragma unroll
                        for (int j = 0; j < 3; ++j) atomicAdd(&gpart[OFF_BR + j], __uint_as_float(r[N_CLASS + j]));
                    } else if (kin >= 0) {                                 // [e | rgb_emb]^T dRGB: rgb_linear.0.weight
#pragma unroll
                        for (int j = 0; j < 3; ++j) atomicAdd(&gpart[OFF_WR + j * D_RGB_IN + kin], __uint_as_float(r[N_CLASS + j]));
                    }
                }
                if (prof && blockIdx.x == 0 && k == 1 && wt == 0) prof[20 + L] = clock64();
                umma::fence_before_sync();
                umma::mbar_arrive(c.bars + B_DWFREE);    // DW fully read: the next layer's first MMA may overwrite it
            }
        }
    } else {
        // =============================== SCATTER ===============================
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(REGS_SCATTER));
        uint32_t k = 0;
        for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++k) {
            const int64_t slot = tile * TC_TP + p;
            const bool valid = slot < N;
            const int64_t i = valid ? am(slot) : 0;
            float x[3] = {0.f, 0.f, 0.f};
            if (valid) src.point(i, f, x);
            c.ok &= umma::mbar_wait_spin(c.bars + B_DG3, k & 1u);
            umma::fence_after_sync();
            if (prof && blockIdx.x == 0 && k == 1 && p == 0) prof[24] = clock64();
            uint32_t r[32];
            umma::tmem_ld32(c.lane_base + T_D + 64, r);
            umma::wait_ld();
            umma::fence_before_sync();
            umma::mbar_arrive(c.bars + B_DCONS);
            // (holding the gradients back until the chain has left the tile -- so that the reductions do not compete with the
            // hand-offs for the load / store unit -- was measured slower: 0.312 vs 0.291 ms; the forward phases of the next tile
            // use the unit just as much)
            if (prof && blockIdx.x == 0 && k == 1 && p == 0) prof[26] = clock64();
#ifndef MF_EXP_NOSCATTER
            if constexpr (is_det_rows<Src>::value) { if (valid) det_store_row(grad_grid, slot, x, r); } else {   // (deterministic mode)
                // (slots behind the end of the list carry an all-zero gradient row: they join the runs with zeros and are skipped)
#pragma unroll 1
                for (int gq = 0; gq < 4; ++gq) {         // rolled over groups of 4 levels: three roles share the instruction cache
                    float dy8[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        dy8[j] = valid ? __uint_as_float(gq == 0 ? r[j] : (gq == 1 ? r[8 + j] : (gq == 2 ? r[16 + j] : r[24 + j]))) : 0.f;
#pragma unroll 1
                    for (int ll = 0; ll < 4; ++ll) {
                        const float2 dy = ll == 0 ? make_float2(dy8[0], dy8[1]) : (ll == 1 ? make_float2(dy8[2], dy8[3]) : (ll == 2 ? make_float2(dy8[4], dy8[5]) : make_float2(dy8[6], dy8[7])));
                        if (agg) grid_level_scatter_agg(x, dy, grad_grid, level_info(f, gq * 4 + ll), tid & 31);
                        else if (valid) { float dx[3]; grid_level_bwd<false>(x, dy, nullptr, grad_grid, level_info(f, gq * 4 + ll), dx); }
                    }
                }
            }
#endif
            if (prof && blockIdx.x == 0 && k == 1 && p == 0) prof[25] = clock64();
        }
    }
#undef B2_MARK
    if (!c.ok && err) atomicExch(err, 1);
    mf_pdl_trigger();                                    // every tile of this CTA is done: the next kernel may start its prologue
    umma::fence_before_sync();
    __syncthreads();
    if (prof && tid == 0 && blockIdx.x < 256) prof[577 + 2 * blockIdx.x] = mf_globaltimer();
    if (warp == 0) umma::tmem_dealloc<512>(c.tmem);
}
