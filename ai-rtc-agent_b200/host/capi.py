"""ctypes binding of libb200sd.so (include/b200sd.h).  There is no CPU fallback: if the shared
library is missing or a call fails this module raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# B200SD_LIB: developer override (e.g. the -DB2_TIMELINE build used by tools/timeline_chain.py)
LIB_PATH = os.environ.get("B200SD_LIB") or os.path.join(os.path.dirname(_HERE), "libb200sd.so")


class B2Error(RuntimeError):
    pass


class ActView(C.Structure):
    _fields_ = [("ptr", C.c_void_p), ("n", C.c_int), ("h", C.c_int), ("w", C.c_int), ("c", C.c_int),
                ("ld", C.c_int)]


class IgemmDesc(C.Structure):
    _fields_ = [
        ("src", ActView * 3), ("ntap", C.c_int * 3), ("nseg", C.c_int),
        ("w", C.c_void_p), ("w_rows", C.c_int), ("w_ld", C.c_int), ("stride", C.c_int),
        ("nb", C.c_int), ("ho", C.c_int), ("wo", C.c_int),
        ("bn", C.c_int), ("splits", C.c_int), ("partial", C.c_void_p),
        ("out", C.c_void_p), ("ldc", C.c_int),
        ("colbias", C.c_void_p), ("colbias_bstride", C.c_int),
        ("res", C.c_void_p), ("ldr", C.c_int),
        ("acc_scale", C.c_float), ("res_scale", C.c_float),
        ("flags", C.c_int), ("n_valid", C.c_int), ("swap", C.c_int),
        ("rowstat_out", C.c_void_p), ("rowstat_in", C.c_void_p), ("colsum", C.c_void_p), ("ln_c", C.c_int), ("ln_eps", C.c_float),
        ("out2", C.c_void_p), ("ld2", C.c_int), ("col2", C.c_int),
    ]


class IgemmPlanInfo(C.Structure):
    _fields_ = [
        ("mode", C.c_int), ("swap", C.c_int), ("bn", C.c_int), ("splits", C.c_int),
        ("grid_x", C.c_int), ("grid_y", C.c_int), ("grid_z", C.c_int),
        ("num_stages", C.c_int), ("acc_bufs", C.c_int), ("total_kb", C.c_int), ("kb_per_split", C.c_int),
        ("tmem_cols", C.c_int), ("m_tiles", C.c_int),
        ("smem_bytes", C.c_int64), ("rows_total", C.c_int64),
    ]


class AttnDesc(C.Structure):
    _fields_ = [
        ("q", C.c_void_p), ("ldq", C.c_int),
        ("k", C.c_void_p), ("ldk", C.c_int), ("k_bstride", C.c_int64), ("k_rows", C.c_int64),
        ("vt", C.c_void_p), ("ldvt", C.c_int), ("vt_bstride", C.c_int64), ("vt_cols", C.c_int64),
        ("out", C.c_void_p), ("ldo", C.c_int),
        ("nb", C.c_int), ("heads", C.c_int), ("sq", C.c_int), ("skv", C.c_int), ("d_real", C.c_int),
        ("dp", C.c_int),
    ]


class EngineConfig(C.Structure):
    _fields_ = [
        ("block_out_channels", C.c_int * 4), ("heads", C.c_int * 4), ("down_attn", C.c_int * 4),
        ("cross_attention_dim", C.c_int), ("layers_per_block", C.c_int), ("norm_groups", C.c_int),
        ("ctx_tokens", C.c_int), ("batch", C.c_int), ("height", C.c_int), ("width", C.c_int),
        ("do_add_noise", C.c_int), ("use_cuda_graph", C.c_int),
    ]


IN_U8_NHWC, IN_F32_NCHW, IN_F16_NCHW = 0, 1, 2
OUT_U8_NCHW, OUT_F16_NCHW = 0, 1
IG_RELU = 1
IG_GEGLU = 2
IG_TCONV = 64
IG_PAIR = 128
CFG_NONE, CFG_SELF, CFG_INITIALIZE, CFG_FULL = 0, 1, 2, 3
CFG_TYPES = {"none": CFG_NONE, "self": CFG_SELF, "initialize": CFG_INITIALIZE, "full": CFG_FULL}

_lib = None


def lib() -> C.CDLL:
    """Load libb200sd.so; fails loudly when it has not been built (python __graft_entry__.py)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise B2Error(f"{LIB_PATH} not found: build it with `make -C ai-rtc-agent_b200/csrc` "
                          "(or __graft_entry__.build()); there is no CPU fallback")
        _lib = C.CDLL(LIB_PATH)
        _lib.b2sd_last_error.restype = C.c_char_p
        _lib.b2sd_version.restype = C.c_int
        _lib.b2sd_op_igemm.argtypes = [C.POINTER(IgemmDesc), C.c_void_p]
        _lib.b2sd_op_igemm.restype = C.c_int
        _lib.b2sd_igemm_plan_dry.argtypes = [C.POINTER(IgemmDesc), C.c_int, C.c_int, C.POINTER(IgemmPlanInfo)]
        _lib.b2sd_igemm_plan_dry.restype = C.c_int
        _lib.b2sd_groupnorm_plan_dry.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
        _lib.b2sd_groupnorm_plan_dry.restype = C.c_int
        _lib.b2sd_igemm_partial_floats.argtypes = [C.c_int, C.c_int64, C.c_int]
        _lib.b2sd_igemm_partial_floats.restype = C.c_uint64
        vp, ci, cf, i64 = C.c_void_p, C.c_int, C.c_float, C.c_int64
        _lib.b2sd_op_attention.argtypes = [C.POINTER(AttnDesc), vp]
        _lib.b2sd_op_groupnorm.argtypes = [vp, ci, ci, vp, ci, ci, vp, vp, vp, ci, ci, ci, ci, cf, ci, vp]
        _lib.b2sd_op_layernorm.argtypes = [vp, ci, vp, vp, vp, ci, i64, ci, cf, vp]
        _lib.b2sd_op_upsample2x.argtypes = [vp, vp, ci, ci, ci, ci, vp]
        _lib.b2sd_op_smallconv.argtypes = [vp, vp, vp, vp, ci, ci, ci, ci, ci, ci, ci, ci, ci, vp]
        _lib.b2sd_op_lcm_step.argtypes = [vp, vp, vp, vp, vp, ci, ci, ci, vp]
        _lib.b2sd_op_lcm_cfg_step.argtypes = [vp, vp, vp, vp, vp, vp, ci, ci, ci, ci, cf, cf, vp]
        _lib.b2sd_op_post_u8.argtypes = [vp, ci, vp, ci, ci, ci, vp]
        _lib.b2sd_op_nv12_to_rgb.argtypes = [vp, ci, vp, ci, vp, ci, ci, ci, vp]
        _lib.b2sd_op_rgb_to_nv12.argtypes = [vp, vp, ci, vp, ci, ci, ci, ci, vp]
        _lib.b2sd_codec_probe.restype = C.c_int
        _lib.b2sd_create.argtypes = [C.POINTER(EngineConfig), C.POINTER(vp)]
        _lib.b2sd_destroy.argtypes = [vp]
        _lib.b2sd_create_lane.argtypes = [vp, C.POINTER(EngineConfig), C.POINTER(vp)]
        _lib.b2sd_load_tensor.argtypes = [vp, C.c_char_p, vp, ci, C.POINTER(i64), ci]
        _lib.b2sd_prepare.argtypes = [vp, vp, vp, vp, vp, vp]
        _lib.b2sd_export_packed.argtypes = [vp, C.c_char_p]
        _lib.b2sd_import_packed.argtypes = [vp, C.c_char_p]
        _lib.b2sd_set_prompt_embeds.argtypes = [vp, vp, vp]
        _lib.b2sd_set_timesteps.argtypes = [vp, vp, vp]
        _lib.b2sd_set_guidance.argtypes = [vp, ci, cf, cf, vp]
        _lib.b2sd_step.argtypes = [vp, vp, ci, ci, vp, vp]
        _lib.b2sd_step_ex.argtypes = [vp, vp, ci, ci, ci, vp, ci, vp]
        _lib.b2sd_get_tensor.argtypes = [vp, C.c_char_p, vp, i64, C.POINTER(i64), C.POINTER(ci), vp]
        _lib.b2sd_launches_per_step.argtypes = [vp]
        _lib.b2sd_share_stream_state.argtypes = [vp, vp]
        _lib.b2sd_share_stream_state.restype = C.c_int
        _lib.b2sd_set_concurrency.argtypes = [vp, ci]
        _lib.b2sd_set_concurrency.restype = C.c_int
        _lib.b2sd_profile.argtypes = [vp, vp, ci, ci, vp, ci, C.c_char_p, i64, vp]
        _lib.b2sd_profile.restype = C.c_int
        _lib.b2sd_profile_kind.argtypes = [vp, C.c_char_p, ci, C.POINTER(C.c_double), C.POINTER(ci), C.POINTER(C.c_double), vp]
        _lib.b2sd_profile_kind.restype = C.c_int
        _lib.b2sd_profile_gate.argtypes = [ci]
        _lib.b2sd_profile_gate.restype = C.c_int
        for name in ("create", "create_lane", "destroy", "load_tensor", "prepare", "export_packed", "import_packed", "set_prompt_embeds", "set_timesteps",
                     "set_guidance", "step",
                     "step_ex", "get_tensor", "launches_per_step"):
            getattr(_lib, "b2sd_" + name).restype = C.c_int
        for name in ("attention", "groupnorm", "layernorm", "upsample2x", "smallconv", "lcm_step", "lcm_cfg_step", "post_u8", "nv12_to_rgb", "rgb_to_nv12"):
            getattr(_lib, "b2sd_op_" + name).restype = C.c_int
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise B2Error(f"{what}: {lib().b2sd_last_error().decode(errors='replace')}")


def current_stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
