// Launch helper choosing between the tcgen05 decoder (default) and the fp32 CUDA-core decoder.
#pragma once
#include "field_launch.cuh"
#include "field_tc.cuh"
#include "field_tc2.cuh"
#include "field_tc3.cuh"

template <class Src, class Epi, bool SDF_ONLY>
static inline int launch_field_fwd_tc(const FieldDev& d, const Src& src, const Epi& epi, int64_t N, cudaStream_t st,
                                      const unsigned int* n_dev = nullptr) {
    int rc = set_smem(field_fwd_tc_kernel<Src, Epi, SDF_ONLY>, SMEM_TC); if (rc) return rc;
    const int64_t tiles = (N + TC_TP - 1) / TC_TP;
    const int64_t cap = mf_sm_count_cached();
    const int grid = (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
    field_fwd_tc_kernel<Src, Epi, SDF_ONLY><<<grid, TC_NT, SMEM_TC, st>>>(d, src, epi, N, n_dev, d.tc_img, mf_tc_error_flag(), mf_tc_profile_buffer());
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// dual-pipeline kernel: two 128-point tiles in flight per CTA
template <class Src, class Epi, bool SDF_ONLY>
static inline int launch_field_fwd_tc2(const FieldDev& d, const Src& src, const Epi& epi, int64_t N, cudaStream_t st,
                                       const unsigned int* n_dev = nullptr) {
    int rc = set_smem(field_fwd_tc2_kernel<Src, Epi, SDF_ONLY>, SMEM_TC2); if (rc) return rc;
    const int64_t pairs = ((N + TC_TP - 1) / TC_TP + 1) / 2;
    const int64_t cap = mf_sm_count_cached();
    const int grid = (int)(pairs < cap ? (pairs > 0 ? pairs : 1) : cap);
    field_fwd_tc2_kernel<Src, Epi, SDF_ONLY><<<grid, 2 * T2_GT, SMEM_TC2, st>>>(d, src, epi, N, n_dev, d.tc_img, mf_tc_error_flag());
    MF_LAUNCH_CHECK();
    return MF_OK;
}

// producer / consumer kernel: gather warps feed decoder warps through tensor memory
template <class Src, class Epi, bool SDF_ONLY>
static inline int launch_field_fwd_tc3(const FieldDev& d, const Src& src, const Epi& epi, int64_t N, cudaStream_t st,
                                       const unsigned int* n_dev = nullptr) {
    int rc = set_smem(field_fwd_tc3_kernel<Src, Epi, SDF_ONLY>, SMEM_TC3); if (rc) return rc;
    const int64_t tiles = (N + TC_TP - 1) / TC_TP;
    const int64_t cap = mf_sm_count_cached() - mf_sm_reserve() > 0 ? mf_sm_count_cached() - mf_sm_reserve() : 1;
    const int grid = (int)(tiles < cap ? (tiles > 0 ? tiles : 1) : cap);
    MF_CUDA(mf_launch(field_fwd_tc3_kernel<Src, Epi, SDF_ONLY>, grid, 2 * T3_GT, SMEM_TC3, st, d, src, epi, N, n_dev, d.tc_img,
                      mf_tc_error_flag(), mf_tc_profile_buffer(), mf_tile_counter()));
    return MF_OK;
}

template <class Src, class Epi, bool SDF_ONLY>
static inline int launch_field_fwd_auto_(const FieldDev& d, const Src& src, const Epi& epi, int64_t N, cudaStream_t st,
                                         const unsigned int* n_dev, bool short_launches);

// ktimer_slot >= 0: bracket the kernel with the diagnostic event pair of that slot (mf_debug_kernel_timer)
template <class Src, class Epi, bool SDF_ONLY>
static inline int launch_field_fwd_auto(const FieldDev& d, const Src& src, const Epi& epi, int64_t N, cudaStream_t st,
                                        const unsigned int* n_dev = nullptr, bool short_launches = false, int ktimer_slot = -1) {
    if (ktimer_slot >= 0) mf_ktimer_begin(ktimer_slot, st);
    const int rc = launch_field_fwd_auto_<Src, Epi, SDF_ONLY>(d, src, epi, N, st, n_dev, short_launches);
    if (ktimer_slot >= 0) mf_ktimer_end(ktimer_slot, st);
    return rc;
}

template <class Src, class Epi, bool SDF_ONLY>
static inline int launch_field_fwd_auto_(const FieldDev& d, const Src& src, const Epi& epi, int64_t N, cudaStream_t st,
                                         const unsigned int* n_dev, bool short_launches) {
    // short launches (a few tiles per CTA, e.g. the per-submap chunks of the joint query) cannot fill the
    // producer -> consumer pipeline; two independent tiles per CTA (dual pipeline) serve them better
    if (d.impl == 0 && short_launches) return launch_field_fwd_tc2<Src, Epi, SDF_ONLY>(d, src, epi, N, st, n_dev);
    if (d.impl == 0) return launch_field_fwd_tc3<Src, Epi, SDF_ONLY>(d, src, epi, N, st, n_dev);
    if (d.impl == 3) return launch_field_fwd_tc2<Src, Epi, SDF_ONLY>(d, src, epi, N, st, n_dev);   // dual pipeline (A/B)
    if (d.impl == 2) return launch_field_fwd_tc<Src, Epi, SDF_ONLY>(d, src, epi, N, st, n_dev);   // single pipeline (A/B)
    return launch_field_fwd<Src, Epi, SDF_ONLY>(d, src, epi, N, st, n_dev);
}
