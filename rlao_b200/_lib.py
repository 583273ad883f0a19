"""ctypes binding of libaoenv_b200.so (include/aoenv.h).

There is no CPU fallback: if the shared library is missing the import of any compute path raises
`AOEnvLibraryError` telling the user how to build it (`python -c "import __graft_entry__ as g; g.build()"`
or `bash rlao_b200/csrc/build.sh`).
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libaoenv_b200.so")


class AOEnvLibraryError(RuntimeError):
    pass


class DetectorStruct(C.Structure):
    """aoenv_detector_t (include/aoenv.h)."""
    _fields_ = [
        ("photon_noise", C.c_int32), ("sensor_emccd", C.c_int32), ("has_fwc", C.c_int32), ("bits", C.c_int32),
        ("qe", C.c_float), ("dark_electrons", C.c_float), ("fwc", C.c_float), ("gain", C.c_float),
        ("readout_noise", C.c_float), ("reserved", C.c_uint32), ("seed", C.c_uint64), ("frame_counter", C.c_uint64),
    ]


class DmSepStruct(C.Structure):
    """aoenv_dm_sep_t (include/aoenv.h)."""
    _fields_ = [
        ("rows", C.c_void_p), ("wlr", C.c_void_p), ("ilr", C.c_void_p),
        ("nActP", C.c_int32), ("WL", C.c_int32), ("t_rows", C.c_int32), ("reserved", C.c_int32),
    ]


MAX_LAYERS = 8          # AOENV_MAX_LAYERS (include/aoenv.h)


class LayerState(C.Structure):
    """aoenv_layer_state_t (include/aoenv.h)."""
    _fields_ = [
        ("ratio", C.c_double * 2), ("buff", C.c_double * 2), ("vX", C.c_double), ("vY", C.c_double),
        ("events", C.c_uint64), ("philox_seed", C.c_uint64),
        ("not_done_once", C.c_int32), ("cur", C.c_int32), ("org", C.c_int32 * 2),
    ]


class ShStepStruct(C.Structure):
    """aoenv_sh_step_t (include/aoenv.h)."""
    _fields_ = [(k, C.c_int32) for k in ("B", "nS", "n", "nV", "lds", "nA", "nAct", "nAct2", "ldc", "ldr", "W", "rec_parts",
                                         "use_tc", "geometric")] + [
        ("phase_scale", C.c_float), ("inv_units", C.c_float), ("threshold_cog", C.c_float), ("leak", C.c_float),
        ("n_pupil", C.c_double)] + [(k, C.c_void_p) for k in ("pupil", "amp", "valid", "order", "valid_idx", "ref_xy", "frame",
                                                              "envmax", "stats", "slopes", "slope_planes")] + [
        ("dm", DmSepStruct)] + [(k, C.c_void_p) for k in ("rec_planes", "rec_f32", "rec", "act_idx", "dm_prev", "act_pos",
                                                           "wx", "j0x")]


class AtmState(C.Structure):
    """aoenv_atm_state_t (include/aoenv.h): the per-layer bookkeeping of Atmosphere.update(), shared with the library."""
    _fields_ = [(k, C.c_int32) for k in ("nLayer", "B", "R", "M", "Mc", "pitch", "S", "nI", "nO", "ldz", "ldx", "group_max",
                                         "parts", "fp_off", "warp_kernel", "use_tc")] + [
        ("env_stride", C.c_int64), ("env_offset", C.c_uint64), ("sampling_time", C.c_double), ("ps_loop", C.c_double),
        ("opd_scale", C.c_float), ("reserved", C.c_float), ("weight", C.c_float * MAX_LAYERS),
        ("maps", (C.c_void_p * 2) * MAX_LAYERS), ("ext", C.c_void_p * MAX_LAYERS), ("inner_rc", C.c_void_p),
        ("zx", C.c_void_p), ("zx_planes", C.c_void_p), ("X", C.c_void_p), ("flag", C.c_void_p), ("w_f32", C.c_void_p),
        ("layer", LayerState * MAX_LAYERS),
    ]

_vp, _i, _f, _u64, _d, _i64 = C.c_void_p, C.c_int, C.c_float, C.c_uint64, C.c_double, C.c_int64

# name -> argtypes, exactly the prototypes of include/aoenv.h
PROTOTYPES = {
    "aoenv_atm_gather": [_vp, _i, _i, _i, _i64, _i, _i, _vp, _i, _i, _vp, _u64, _u64, _vp, _i, _vp, _i, _vp],
    "aoenv_atm_ring": [_vp, _i, _i, _i, _i64, _i64, _i, _vp, _i, _vp, _vp, _i, _vp],
    "aoenv_atm_gather_multi": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i64, _vp, _i, _i, _vp, _vp, _i, _vp, _i, _vp],
    "aoenv_atm_ring_multi": [_vp, _vp, _vp, _i, _i, _i, _i, _i64, _i, _vp, _i, _vp, _i, _vp],
    "aoenv_atm_gather_envs": [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i64, _vp, _i, _i, _vp, _i, _vp, _i, _vp],
    "aoenv_atm_ring_envs": [_vp, _vp, _vp, _i, _vp, _i, _i, _i, _i, _i64, _i, _vp, _i, _vp, _vp],
    "aoenv_atm_compact": [_vp, _vp, _i, _i, _i, _i64, _vp, _i64, _vp],
    "aoenv_vk_screens": [_u64, C.c_uint32, _i, _i, _vp, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp, _i,
                         _vp, _i, _i64, _vp],
    "aoenv_vk_screens_envs": [_u64, C.c_uint32, _vp, _i, _i, _vp, _vp, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _vp,
                              _i, _vp, _i, _i64, _vp],
    "aoenv_atm_update": [_vp, _vp, _vp, _vp],
    "aoenv_sh_step": [_vp, _i] + [_vp] * 12,
    "aoenv_atm_phase": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _vp],
    "aoenv_atm_phase_envs": [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp, _vp, _vp, _vp, _vp, _f, _vp, _i, _vp, _vp],
    "aoenv_gemm_tn": [_vp, _i, _vp, _i, _vp, _i, _i, _i, _i, _f, _vp],
    "aoenv_split_bf16": [_vp, _i, _i, _i, _i, _vp, _i, _vp],
    "aoenv_gemm_tn_tc": [_vp, _vp, _i, _i, _vp, _i, _i, _i, _i, _f, _vp],
    "aoenv_dm_surface_separable": [_vp, _i, _vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _vp, _vp],
    "aoenv_set_wfs6_variant": [_i],
    "aoenv_detector_integrate": [_vp, _i, _i, _i, _vp, _vp],
    "aoenv_shwfs_camera": [_vp, _vp, _i, _i, _i, _vp, _i, _vp, _vp],
    "aoenv_shwfs_frame": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp, _i, _vp, _vp, _vp, _vp],
    "aoenv_shwfs_frame_dm": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _f, _vp, _i, _vp, _vp, _vp, _vp],
    "aoenv_shwfs_slopes": [_vp, _vp, _i, _vp, _i, _vp, _f, _f, _i, _i, _i, _vp, _i, _vp, _i, _vp],
    "aoenv_shwfs_fused": [_vp, _vp, _vp, _vp, _f, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _i, _f, _f, _vp, _vp, _i, _vp, _i,
                          _vp, _vp, _vp],
    "aoenv_shwfs_fused_smem": [_i, _i, _i, _i, _i, _i],
    "aoenv_dm_rows": [_vp, _i, _vp, _i, _i, _i, _vp, _vp, _i, _i, _i, _vp, _vp],
    "aoenv_shwfs_geometric": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _i, _vp, _i, _vp, _vp],
    "aoenv_shwfs_geometric_f64": [_vp, _vp, _vp, _i, _i, _i, _i, _d, _d, _vp, _i, _vp],
    "aoenv_shwfs_measure_f64": [_vp, _vp, _vp, _vp, _vp, _i, _vp, _d, _d, _i, _i, _i, _d, _i, _vp, _vp, _vp, _i, _vp],
    "aoenv_normal_fill": [_u64, _u64, _i, _i, _i, _f, _vp, _vp, _i, _vp],
    "aoenv_vec_to_img": [_vp, _i, _vp, _i, _i, _i, _f, _vp, _vp],
    "aoenv_pyramid_supported": [_i],
    "aoenv_pyramid_frames": [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _vp, _vp, _vp, _vp],
    "aoenv_command_update": [_vp, _vp, _i, _i, _i, _f, _vp, _vp, _i, _vp],
    "aoenv_observe": [_vp, _i, _vp, _i, _i, _i, _vp, _d, _f, _vp, _vp, _vp, _vp, _vp, _vp],
    "aoenv_psf_image": [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _i, _vp, _vp, _vp, _vp, _vp, _vp],
    "aoenv_psf_peak": [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _vp, _i, _vp, _vp, _vp, _vp],
}

_lib = None


def load():
    """Loads the shared library (once) and declares every prototype."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AOEnvLibraryError(
            f"{LIB_PATH} not found: the CUDA extension has not been built. Build it with "
            "`bash rlao_b200/csrc/build.sh` (needs nvcc with sm_100a support). rlao_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.aoenv_abi_version.restype = C.c_int
    lib.aoenv_last_error.restype = C.c_char_p
    lib.aoenv_launch_count.restype = C.c_uint64
    lib.aoenv_set_pdl.argtypes, lib.aoenv_set_pdl.restype = [C.c_int], C.c_int
    for name, args in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.argtypes = args
        fn.restype = C.c_int
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        raise RuntimeError(f"libaoenv_b200 {what} failed ({rc}): {load().aoenv_last_error().decode()}")


def ptr(t):
    """Device (or host) address of a tensor, or NULL."""
    return None if t is None else t.data_ptr()          # plain int: ctypes converts it for a c_void_p parameter


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_ptr(device=None):
    """cudaStream_t of torch's current stream on `device` (called before every C-ABI launch: the raw accessor is ~20x
    cheaper than building a torch.cuda.Stream object)."""
    if _raw_stream is not None:
        if device is None:
            idx = torch.cuda.current_device()
        else:
            idx = device.index if isinstance(device, torch.device) else torch.device(device).index
            if idx is None:
                idx = torch.cuda.current_device()
        return _raw_stream(idx)
    return torch.cuda.current_stream(device).cuda_stream


def launch_count():
    return int(load().aoenv_launch_count())


def require_cuda(device):
    if not torch.cuda.is_available():
        raise AOEnvLibraryError("rlao_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    dev = torch.device(device if device is not None else "cuda:0")
    if dev.type != "cuda":
        raise AOEnvLibraryError(f"rlao_b200 objects live on CUDA devices, got {dev}")
    return dev
