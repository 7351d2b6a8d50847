"""ctypes binding of librsdf_b200.so (the C ABI declared in include/rsdf_b200.h).

There is NO fallback: if the shared library is missing or a launch fails, a RuntimeError is
raised.  Tensors cross the boundary as raw device pointers + the current CUDA stream.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("RSDF_LIB_PATH") or os.path.join(_HERE, "librsdf_b200.so")   # override: developer experiments
_lib = None

c_p, c_i, c_f = ctypes.c_void_p, ctypes.c_int, ctypes.c_float

MAX_LEVELS = 32


class HashGridMetaC(ctypes.Structure):
    _fields_ = [("n_levels", ctypes.c_int32), ("n_features", ctypes.c_int32),
                ("scale", ctypes.c_float * MAX_LEVELS), ("res", ctypes.c_uint32 * MAX_LEVELS),
                ("offset", ctypes.c_uint32 * (MAX_LEVELS + 1))]


class SdfMlpC(ctypes.Structure):
    _fields_ = [("w1_blob", c_p), ("w2_blob", c_p), ("w3_blob", c_p), ("b1", c_p), ("b2", c_p), ("b3", c_p),
                ("w3_row0", c_p), ("n_in", ctypes.c_int32), ("n_out", ctypes.c_int32), ("precision", ctypes.c_int32)]


class ReluFwdC(ctypes.Structure):
    _fields_ = [("w", c_p), ("bias", c_p), ("r_pad", ctypes.c_int32), ("r_real", ctypes.c_int32),
                ("k_pad", ctypes.c_int32), ("n_samples", ctypes.c_int32), ("inp", c_p * 3), ("in_w", ctypes.c_int32 * 3),
                ("in_scale", ctypes.c_float * 3), ("in_shift", ctypes.c_float * 3), ("n_in", ctypes.c_int32),
                ("a_in", c_p), ("a0_save", c_p), ("a_out", c_p), ("rows_out", c_p), ("fp16", ctypes.c_int32)]


class ReluBwdC(ctypes.Structure):
    _fields_ = [("w", c_p), ("r_pad", ctypes.c_int32), ("r_real", ctypes.c_int32), ("k_pad", ctypes.c_int32),
                ("k_real", ctypes.c_int32), ("n_samples", ctypes.c_int32), ("zb_in", c_p), ("g_rows", c_p),
                ("amax", c_p), ("a_in", c_p), ("zb_out", c_p), ("rows_out", c_p * 3), ("seg_w", ctypes.c_int32 * 3),
                ("seg_scale", ctypes.c_float * 3), ("first_layer", ctypes.c_int32), ("gW", c_p), ("gb_prev", c_p),
                ("gb_self", c_p), ("fp16", ctypes.c_int32)]


class SplitShadeC(ctypes.Structure):
    _fields_ = [("raw_albedo", c_p), ("raw_roughness", c_p), ("raw_metallic", c_p), ("raw_env", c_p), ("normals", c_p),
                ("dirs", c_p), ("fg_lut", c_p), ("lut_h", ctypes.c_int32), ("lut_w", ctypes.c_int32), ("diffuse", c_p),
                ("diffuse_res", ctypes.c_int32), ("specular_levels", c_p), ("specular_res", c_p),
                ("n_levels", ctypes.c_int32), ("min_roughness", ctypes.c_float), ("max_roughness", ctypes.c_float),
                ("stage", ctypes.c_int32), ("n", ctypes.c_int32)]


ADAM_MAX_GROUPS = 8


class AdamGroupsC(ctypes.Structure):
    _fields_ = [("n_groups", ctypes.c_int32), ("end", ctypes.c_int64 * ADAM_MAX_GROUPS),
                ("step_size", ctypes.c_float * ADAM_MAX_GROUPS), ("one_minus_beta1", ctypes.c_float * ADAM_MAX_GROUPS),
                ("beta2", ctypes.c_float * ADAM_MAX_GROUPS), ("one_minus_beta2", ctypes.c_float * ADAM_MAX_GROUPS),
                ("eps", ctypes.c_float * ADAM_MAX_GROUPS),
                ("bias2_sqrt", ctypes.c_float * ADAM_MAX_GROUPS), ("weight_decay", ctypes.c_float * ADAM_MAX_GROUPS),
                ("skip", ctypes.c_int32 * ADAM_MAX_GROUPS)]


# name -> argtypes (restype is int for all but the two string getters)
_SIGS = {
    "rsdf_ray_aabb_intersect": [c_p, c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_grid_pack_bits": [c_p, c_i, c_p, c_p],
    "rsdf_march_count": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_f, c_i, c_p, c_p, c_p, c_p],
    "rsdf_march_fill": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_f, c_i, c_p, c_p, c_p, c_p, c_p],
    "rsdf_march_count_keep": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_f, c_f, c_i, c_p, c_p, c_p, c_p, c_i, c_p],
    "rsdf_march_compact": [c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p],
    "rsdf_grid_query": [c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_p],
    "rsdf_pack_info": [c_p, c_i, c_i, c_p, c_p],
    "rsdf_weight_from_alpha_fwd": [c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_weight_from_alpha_bwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p],
    "rsdf_accumulate_fwd": [c_p, c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_accumulate_bwd": [c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p],
    "rsdf_neus_render_fwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_i, c_p, c_p, c_p, c_p, c_p],
    "rsdf_neus_render_bwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_i,
                             c_p, c_p, c_p, c_p, c_p],
    "rsdf_split_render_fwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_f, c_i, c_p, c_p, c_p, c_p, c_p],
    "rsdf_split_render_bwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_f, c_i,
                              c_p, c_p, c_p, c_p, c_p],
    "rsdf_sdf_reg_fwd": [c_p, c_p, c_i, c_f, c_p, c_p, c_p],
    "rsdf_sdf_reg_bwd": [c_p, c_p, c_i, c_f, c_p, c_p, c_p, c_p],
    "rsdf_sample_setup": [c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p, c_p],
    "rsdf_normalize3_fwd": [c_p, c_i, c_f, c_p, c_p],
    "rsdf_normalize3_bwd": [c_p, c_p, c_i, c_f, c_p, c_p],
    "rsdf_hashgrid_fwd": [c_p, c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_hashgrid_bwd_table": [c_p, c_p, c_p, c_i, c_p, c_p],
    "rsdf_hashgrid_bwd_input": [c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_hashgrid_bwd_bwd": [c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_p],
    "rsdf_hashgrid_fd6": [c_p, c_p, c_p, c_i, c_f, c_f, c_p, c_p, c_p],
    "rsdf_hashgrid_bwd_table2": [c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p],
    "rsdf_hashgrid_jvp": [c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_sh_fwd": [c_p, c_i, c_i, c_p, c_p],
    "rsdf_sh_bwd": [c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_tex2d_fwd": [c_p, c_i, c_i, c_i, c_i, c_p, c_i, c_p, c_p],
    "rsdf_tex2d_bwd": [c_p, c_i, c_i, c_i, c_i, c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_cube_sample_fwd": [c_p, c_p, c_i, c_p, c_p, c_i, c_p, c_p],
    "rsdf_cube_sample_bwd": [c_p, c_p, c_p, c_i, c_p, c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_split_shade_fwd": [c_p, c_p, c_p],
    "rsdf_split_shade_bwd": [c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "rsdf_cubemap_texel_table": [c_i, c_p, c_p],
    "rsdf_diffuse_cubemap": [c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_specular_bounds": [c_p, c_i, c_f, c_p, c_p, c_p],
    "rsdf_specular_cubemap": [c_p, c_p, c_p, c_i, c_f, c_f, c_i, c_p, c_p],
    "rsdf_specular_build": [c_p, c_p, c_p, c_i, c_f, c_f, c_i, c_p, c_p, c_p],
    "rsdf_specular_apply": [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_mlp_pack_weight": [c_p, c_i, c_i, c_i, c_i, c_p, c_p],
    "rsdf_mlp_fwd": [c_p, c_p],
    "rsdf_mm_stream": [c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_i, c_p],
    "rsdf_mm_tn": [c_p, c_p, c_p, c_i, c_i, c_i, c_p],
    "rsdf_sdf_mlp_fwd": [c_p, c_p, c_i, c_f, c_f, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p],
    "rsdf_sdf_mlp_bwd": [c_p, c_p, c_i, c_f, c_f, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p, c_p,
                         c_p, c_p, c_p, c_p, c_p],
    "rsdf_sdf_mlp_eval": [c_p, c_p, c_i, c_f, c_f, c_p, c_i, c_i, c_p, c_p],
    "rsdf_absmax2": [c_p, ctypes.c_longlong, c_p, ctypes.c_longlong, c_p, c_i, c_p],
    "rsdf_relu_layer_fwd": [c_p, c_p],
    "rsdf_relu_layer_bwd": [c_p, c_p],
    "rsdf_adam_step": [c_p, c_p, c_p, c_p, ctypes.c_longlong, c_p, c_i, c_p],
    "rsdf_freq_encode_fwd": [c_p, c_i, c_i, c_i, c_f, c_f, c_p, c_p, c_p],
    "rsdf_freq_encode_bwd": [c_p, c_p, c_i, c_i, c_i, c_f, c_f, c_p, c_p, c_p],
    "rsdf_get_rays": [c_p, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_p, c_p],
    "rsdf_composite_fwd": [c_p, c_p, c_p, c_i, c_i, c_p, c_p],
    "rsdf_composite_bwd": [c_p, c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p],
    "rsdf_neus_loss_fwd": [c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_neus_loss_bwd": [c_p, c_p, c_p, c_p, c_p, c_i, c_p, c_p, c_p],
    "rsdf_occ_points": [c_p, c_p, ctypes.c_longlong, c_i, c_p, c_p, c_p],
    "rsdf_occ_update": [c_p, c_p, c_p, c_p, ctypes.c_longlong, c_f, c_p],
    "rsdf_occ_threshold": [c_p, ctypes.c_longlong, c_f, c_p, c_p, c_p, c_p],
    "rsdf_neus_alpha": [c_p, c_p, c_p, c_p, c_p, c_f, c_i, c_p, c_p],
    "rsdf_vis_round_lens": [c_p, c_p, c_i, c_i, c_f, c_i, ctypes.c_longlong, c_p, c_p],
    "rsdf_vis_round_fill": [c_p, c_p, c_p, c_i, c_i, c_p, c_p, c_p, c_p, c_p, c_p, c_p],
    "rsdf_vis_round_scatter": [c_p, c_p, ctypes.c_longlong, ctypes.c_longlong, c_p, c_p, c_p],
    "rsdf_tc_gemm_test": [c_i, c_p, c_p, c_p, c_p, c_i, c_i, c_i, c_i, c_i, c_i, c_p],
    "rsdf_mc_count": [c_p, c_i, c_i, c_i, c_f, c_i, c_p, c_p, c_p],
    "rsdf_mc_emit": [c_p, c_i, c_i, c_i, c_f, c_i, c_p, c_p, c_p, c_p],
}


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -m rise_sdf_b200.build` "
                "(there is no CPU / PyTorch fallback for the hot path)")
        L = ctypes.CDLL(LIB_PATH)
        L.rsdf_version.restype = ctypes.c_char_p
        L.rsdf_error_string.restype = ctypes.c_char_p
        L.rsdf_error_string.argtypes = [c_i]
        for name, args in _SIGS.items():
            fn = getattr(L, name)
            fn.argtypes = args
            fn.restype = c_i
        _lib = L
    return _lib


def exported_symbols():
    return ["rsdf_version", "rsdf_error_string"] + list(_SIGS)


def ptr(t):
    """Device pointer of a contiguous tensor (None -> NULL)."""
    if t is None:
        return None
    assert t.is_contiguous(), "rsdf ops need contiguous tensors"
    if t.is_cuda and t.device.index != torch.cuda.current_device():
        # launches go to torch.cuda.current_stream() of the CURRENT device: a tensor living elsewhere would be an
        # illegal access, not an error (one process per GPU sets the device once: bench.py, tests)
        raise RuntimeError(f"tensor on {t.device} but the current CUDA device is {torch.cuda.current_device()}: "
                           "call torch.cuda.set_device() (one process per GPU) before using rise_sdf_b200")
    return t.data_ptr()


def stream():
    return torch.cuda.current_stream().cuda_stream


# kernels launched per C-ABI entry point (for bench.py's gpu_launches count)
LAUNCHES = {"rsdf_march_count": 4, "rsdf_march_count_keep": 4, "rsdf_sdf_reg_fwd": 2, "rsdf_neus_loss_fwd": 2,
            "rsdf_occ_update": 2, "rsdf_occ_threshold": 3, "rsdf_mc_count": 2}
SDF_REG_BLOCKS = 1184
LOSS_BLOCKS = 296
STATS = {"enabled": False, "launches": 0, "timed": set(), "events": {}}


def stats_reset(enabled=True, timed=()):
    """bench.py hook: count launches and (for the entry points in `timed`) bracket each call with
    CUDA events on the launching stream.  Off by default; costs nothing when disabled."""
    STATS.update(enabled=enabled, launches=0, timed=set(timed), events={})


def stats_times_ms():
    """name -> (n_calls, total_ms); call after a device synchronize."""
    return {k: (len(v), sum(a.elapsed_time(b) for a, b in v)) for k, v in STATS["events"].items()}


def call(name, *args):
    if STATS["enabled"]:
        STATS["launches"] += LAUNCHES.get(name, 1)
        if name in STATS["timed"]:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            rc = getattr(lib(), name)(*args)
            b.record()
            STATS["events"].setdefault(name, []).append((a, b))
        else:
            rc = getattr(lib(), name)(*args)
    else:
        rc = getattr(lib(), name)(*args)
    if rc != 0:
        raise RuntimeError(f"{name} failed: {lib().rsdf_error_string(rc).decode()} (code {rc})")


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NotImplementedError("Only support cuda inputs.")  # lib/nerfacc/ray_marching.py:131-132


def host6(t):
    """6 floats on the host (roi / aabb) as a ctypes array."""
    vals = [float(v) for v in (t.detach().cpu().tolist() if isinstance(t, torch.Tensor) else t)]
    return (ctypes.c_float * 6)(*vals)
