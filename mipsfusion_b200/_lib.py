"""ctypes binding of the C-ABI shared library (include/mipsfusion_b200.h).

The library is the product: there is no CPU or PyTorch fallback.  ``lib()`` raises
if ``libmipsfusion_b200.so`` has not been built (``python -c "import __graft_entry__ as g; g.build()"``
or ``make -C mipsfusion_b200/csrc``).
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MIPSFUSION_B200_LIB") or os.path.join(_HERE, "libmipsfusion_b200.so")      # (override: A/B builds)
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "mipsfusion_b200.h")

MF_MAX_LEVELS = 16
MF_MLP_PARAMS = 36577
MF_RAW_DIM = 10
MF_MAX_SAMPLES = 128          # render_kernels.cu MAX_S


class GridMeta(C.Structure):
    _fields_ = [("n_levels", C.c_int32), ("n_features", C.c_int32), ("log2_hashmap_size", C.c_int32),
                ("base_resolution", C.c_int32), ("scale", C.c_float * MF_MAX_LEVELS),
                ("resolution", C.c_uint32 * MF_MAX_LEVELS), ("size", C.c_uint32 * MF_MAX_LEVELS),
                ("offset", C.c_uint32 * (MF_MAX_LEVELS + 1)), ("hashed", C.c_uint32 * MF_MAX_LEVELS)]


class Field(C.Structure):
    _fields_ = [("grid", C.c_void_p), ("mlp_prep", C.c_void_p), ("norm_a", C.c_double * 3), ("norm_b", C.c_double * 3),
                ("norm_factor", C.c_double), ("decoder_impl", C.c_int32), ("reserved", C.c_int32), ("meta", GridMeta)]


class RenderCfg(C.Structure):
    _fields_ = [("n_samples_d", C.c_int32), ("n_range_d", C.c_int32), ("perturb", C.c_int32), ("rgb_missing_nz", C.c_int32),
                ("trunc", C.c_double), ("sc_factor", C.c_double), ("depth_trunc", C.c_double), ("emd_w", C.c_double)]


class PointSet(C.Structure):
    _fields_ = [("pts", C.c_void_p), ("ax", C.c_void_p), ("ay", C.c_void_p), ("az", C.c_void_p),
                ("nx", C.c_int32), ("ny", C.c_int32), ("nz", C.c_int32)]


class Submap(C.Structure):
    _fields_ = [("field", Field), ("w2l", C.c_float * 12), ("aabb_min", C.c_double * 3), ("aabb_max", C.c_double * 3),
                ("centroid", C.c_float * 3)]


_P, _I, _L, _D = C.c_void_p, C.c_int, C.c_int64, C.c_double

# name -> (restype, argtypes); mirrors include/mipsfusion_b200.h one to one
PROTOTYPES = {
    "mf_last_error": (C.c_char_p, []),
    "mf_abi_version": (_I, []),
    "mf_device_sm_count": (_I, []),
    "mf_set_decoder_impl": (_I, [_I]),
    "mf_get_decoder_impl": (_I, []),
    "mf_set_bwd_impl": (_I, [_I]),
    "mf_set_dynamic_tiles": (_I, [_I]),
    "mf_set_sm_reserve": (_I, [_I]),
    "mf_containment": (_I, [_P, _P, _P, _P, _P, _P, _I, _L, _I, _P, _P, _P]),
    "mf_tc_check_error": (_I, []),
    "mf_debug_umma_linear": (_I, [_P, _P, _P, _I, _I, _P]),
    "mf_debug_umma_dgrad": (_I, [_P, _P, _P, _I, _P]),
    "mf_debug_umma_wgrad": (_I, [_P, _P, _P, _I, _I, _P]),
    "mf_debug_profile": (_I, [_I, _P]),
    "mf_debug_profile_all": (_I, [_P, _I]),
    "mf_debug_kernel_timer": (_I, [_I]),
    "mf_debug_kernel_ms": (_I, [_I, _P]),
    "mf_hashgrid_meta": (_I, [_I, _I, _I, _I, _D, C.POINTER(GridMeta)]),
    "mf_hashgrid_fwd": (_I, [_P, _P, C.POINTER(GridMeta), _P, _P, _L, _P]),
    "mf_hashgrid_bwd": (_I, [_P, _P, _P, C.POINTER(GridMeta), _P, _P, _L, _P]),
    "mf_freq_fwd": (_I, [_P, _P, _I, _I, _L, _P]),
    "mf_freq_bwd": (_I, [_P, _P, _P, _I, _I, _L, _P]),
    "mf_mlp_prep_size": (_L, []),
    "mf_mlp_prepare": (_I, [_P, _P, _P]),
    "mf_mlp_fwd": (_I, [_P, _P, _P, _P, _P, _L, _P]),
    "mf_field_bwd_workspace_size": (_L, [_L, _I]),
    "mf_mlp_grad_workspace_size": (_L, []),
    "mf_mlp_bwd": (_I, [_P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _L, _P]),
    "mf_field_query": (_I, [_P, C.POINTER(Field), _I, _P, _L, _P]),
    "mf_field_query_bwd": (_I, [_P, C.POINTER(Field), _I, _P, _P, _P, _P, _P, _L, _P]),
    "mf_sample_z": (_I, [_P, _P, _P, _P, _P, C.POINTER(RenderCfg), _P, _P, _L, _P]),
    "mf_feat_cache_size": (_L, [_L]),
    "mf_field_query_rays": (_I, [_P, _P, _P, C.POINTER(Field), _P, _P, _L, _I, _P]),
    "mf_field_query_rays_bwd": (_I, [_P, _P, _P, C.POINTER(Field), _P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_render_loss_fwd": (_I, [_P, _P, _P, _P, _P, C.POINTER(RenderCfg), _P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_render_loss_bwd": (_I, [_P, _P, _P, _P, _P, _P, C.POINTER(RenderCfg), _P, _P, _P, _P, _L, _I, _P]),
    "mf_render_loss_bwd_scalars": (_I, [_P, _P, _P, _I, _P, _I, _P, C.POINTER(RenderCfg), _P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_sample_z_ld": (_I, [_P, _I, _P, _P, _P, _P, C.POINTER(RenderCfg), _P, _P, _L, _P]),
    "mf_render_loss_fwd_ld": (_I, [_P, _P, _P, _I, _P, _I, _P, C.POINTER(RenderCfg), _P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_adam_step": (_I, [_P, _P, _P, _P, _L, _D, _D, _D, _D, _D, _I, _I, _P]),
    "mf_adam_step_sharded": (_I, [_P, _I, _I, _L, _L, _L, _P, _P, _L, _D, _D, _D, _D, _D, _I, C.c_uint64, _P]),
    "mf_adam_step_pair": (_I, [_P, _P, _P, _P, _L, _D, _D, _D, _P, _P, _P, _P, _L, _D, _D, _D, _D, _D, _I, _P]),
    "mf_adam_step_multi": (_I, [_I, _P, _P, _P, _P, _P, _D, _D, _D, _D, _D, _I, _I, _P]),
    "mf_sample_pixels_uniform": (_I, [_I, _I, _I, _I, _P, _P, _P]),
    "mf_topk_workspace_size": (_L, [_L]),
    "mf_sample_pixels_topk": (_I, [_P, _P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mf_gen_rays": (_I, [_P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_kf_store": (_I, [_P, _P, _P, _P, _P, _I, _L, _P, _P]),
    "mf_kf_gather_rays": (_I, [_P, _L, _L, _P, _L, _I, _P, _L, _P, _L, _P, _L, _P, _P, _P, _P]),
    "mf_sample_distinct": (_I, [_L, _L, C.c_uint32, _P, _P]),
    "mf_kf_sample_rays": (_I, [_P, _L, _L, _P, _L, _L, _I, _L, _L, _L, C.c_uint32, _P, _P, _P, _P, _P]),
    "mf_frame_sample_rays": (_I, [_P, _P, _P, _I, _I, _L, C.c_uint32, _P, _P, _P, _P]),
    "mf_gen_rays_packed": (_I, [_P, _P, _P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_gen_rays_bwd": (_I, [_P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_gen_rays_packed_bwd": (_I, [_P, _P, _P, _P, _P, _L, _I, _P]),
    "mf_pose_to_c2w": (_I, [_P, _P, _P]),
    "mf_pose_refine_update": (_I, [_P, _P, _P, _P, _P, _D, _D, _I, _P, _P]),
    "mf_track_handoff": (_I, [_P, _P, _P, _P, _P]),
    "mf_ba_pose_init": (_I, [_P, _P, _I, _P, _P, _P]),
    "mf_ba_pose_update": (_I, [_P, _P, _P, _I, _D, _D, _P, _P]),
    "mf_ro_score": (_I, [_P, _P, _P, _P, _P, _P, C.POINTER(Field), _D, _D, _I, _I, _I, _P, _P, _P, _P, _P]),
    "mf_ro_update": (_I, [_P, _P, _P, _I, _D, _P, _P, _P, _P, _P, _P]),
    "mf_ro_update_gathered": (_I, [_P, _I, _I, _D, _P, _P, _P, _P, _P, _P]),
    "mf_ro_update_peer": (_I, [_P, _P, _I, _I, _L, _L, C.c_uint, _I, _I, _D, _P, _P, _P, _P, _P, _P]),
    "mf_joint_query_scratch_size": (_L, [_L]),
    "mf_joint_query_maxdist": (_I, [C.POINTER(PointSet), C.POINTER(Submap), _I, _L, _L, _P, _P]),
    "mf_joint_query_accumulate": (_I, [C.POINTER(PointSet), C.POINTER(Submap), _I, _I, _I, _P, _P, _I, _L, _L, _P, _P, _P, _P, _P]),
    "mf_joint_query_finalize": (_I, [_P, _P, _I, _L, _P, _P]),
    "mf_mcubes_count_workspace_size": (_L, [_L, _L, _L]),
    "mf_mcubes_count": (_I, [_P, _L, _L, _L, C.c_float, C.c_float, _P, _P, _P]),
    "mf_mcubes_mesh_workspace_size": (_L, [_L]),
    "mf_mcubes_mesh": (_I, [_P, _L, _L, _L, C.c_float, _L, _P, _P, _P, _P, _P]),
    "mf_mesh_seen_mask": (_I, [_P, _L, _P, _P, _I, _P, _I, _I, _I, _P, _P]),
    "mf_mesh_face_mask": (_I, [_P, _P, _L, _P, _P]),
    "mf_overlap_points": (_I, [_P, _P, _I, _I, _P, _I, _P, _I, _P, _I, _P, _P, _P]),
    "mf_overlap_loss": (_I, [_P, _P, _I, _I, _P, _I, _P, _I, _I, _D, _P, _P, _P]),
    "mf_overlap_pose_bwd": (_I, [_P, _P, _I, _I, _P, _I, _P, _I, _P, _I, _P, _P, _I, _I, _P, _P, _P, _P]),
}

_lib = None


class MipsFusionB200Error(RuntimeError):
    pass


def load_library(path=LIB_PATH):
    """Open the shared library and bind every symbol the header declares (no CUDA call is made)."""
    if not os.path.exists(path):
        raise MipsFusionB200Error(
            f"{path} is missing: the sm_100a CUDA library has not been built (run __graft_entry__.build()); "
            "there is no CPU fallback")
    dll = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(dll, name)          # AttributeError if the symbol is not exported
        fn.restype, fn.argtypes = res, args
    return dll


def lib():
    global _lib
    if _lib is None:
        _lib = load_library()
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().mf_last_error().decode(errors="replace")
        raise MipsFusionB200Error(f"{what or 'mipsfusion_b200'} failed ({rc}): {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL).  The tensor must be CUDA, contiguous."""
    if t is None:
        return None
    if not t.is_cuda:
        raise MipsFusionB200Error("mipsfusion_b200 kernels need CUDA tensors (no CPU fallback)")
    if not t.is_contiguous():
        raise MipsFusionB200Error("non-contiguous tensor passed to a kernel")
    return t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream():
    """cudaStream_t of torch's current stream on the current device (the raw getter: building a torch.cuda.Stream object
    per call costs several microseconds, and the drop-in training loop is host-bound)."""
    if _raw_stream is not None:
        return _raw_stream(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream


def f32c(t, device=None):
    """fp32, contiguous, on `device` (no copy when already so)."""
    if device is not None and t.device != device:
        t = t.to(device)
    return t.to(torch.float32).contiguous()


def call(name, *args):
    check(getattr(lib(), name)(*args), name)
