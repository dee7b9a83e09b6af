"""ctypes binding of libmfvit.so (include/mfvit.h).  No fallback: if the library is missing or the device is not
sm_100, every entry point raises."""
import ctypes as C
import os
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmfvit.so")

c_f32p = C.c_void_p
c_vp = C.c_void_p
i64 = C.c_int64
i32 = C.c_int32
f32 = C.c_float


class MfvError(RuntimeError):
    pass


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", c_vp), ("B", c_vp), ("C", c_vp), ("C2", c_vp), ("C3", c_vp), ("bias", c_vp), ("aux", c_vp),
        ("M", i64), ("N", i64), ("K", i64), ("G", i64),
        ("lda", i64), ("ldb", i64), ("ldc", i64),
        ("a_gstride", i64), ("b_gstride", i64), ("c_gstride", i64),
        ("aux_ld", i64), ("aux_gstride", i64), ("bias_gstride", i64),
        ("a_mn_major", i32), ("b_mn_major", i32), ("epilogue", i32), ("splits", i32), ("block_n", i32),
        ("dtype_flags", i32), ("cta_group", i32), ("rows_per_cta", i32),
        ("row_sum", c_vp),
        ("ln_gamma", c_vp), ("ln_beta", c_vp), ("ln_mean", c_vp), ("ln_rstd", c_vp), ("ln_eps", f32), ("ln_out_f32", i32),
    ]


_FUSION_FIELDS = ["ln1_w", "ln1_b", "wq", "wk", "wv", "proj_w", "proj_b", "ln2_w", "ln2_b", "head_w", "head_b",
                  "vhead_w", "vhead_b"]


class FusionParams(C.Structure):
    _fields_ = [(n, c_vp * 2) for n in _FUSION_FIELDS]


class FusionGrads(C.Structure):
    _fields_ = [(n, c_vp * 2) for n in _FUSION_FIELDS]


class EmaChunk(C.Structure):
    _fields_ = [("k", c_vp), ("q", c_vp), ("n", i64)]


class LarsTensor(C.Structure):
    _fields_ = [("p", c_vp), ("g", c_vp), ("mu", c_vp), ("shadow_bf16", c_vp), ("shadow_f16", c_vp), ("n", i64),
                ("chunk0", i64), ("trust", i32), ("reserved", i32)]


LARS_CHUNK = 32768  # MFV_LARS_CHUNK


class VitPlan(C.Structure):
    _fields_ = (
        [(n, i64) for n in ["G", "B", "S", "C", "H", "depth", "hidden", "img", "np", "P"]]
        + [("master", c_vp), ("shadow", c_vp), ("shadow16", c_vp), ("grad", c_vp)]
        + [(n, i64) for n in ["off_cls", "off_pos", "off_pe_w", "off_pe_b", "off_norm_w", "off_norm_b", "off_block0",
                              "block_stride", "r_ln1_w", "r_ln1_b", "r_qkv_w", "r_qkv_b", "r_proj_w", "r_proj_b",
                              "r_ln2_w", "r_ln2_b", "r_fc1_w", "r_fc1_b", "r_fc2_w", "r_fc2_b"]]
        + [("images", c_vp * 2)]
        + [(n, c_vp) for n in ["patches", "acc", "x", "xn", "stats", "qkv", "attn_o", "lse", "u", "gact", "tokens"]]
        + [("save_for_backward", i32), ("stop_grad_conv1", i32), ("fwd_f16", i32), ("gact_bf_per_block", i32)]
        + [(n, c_vp) for n in ["patches_bf", "xn_bf", "attn_o_bf", "gact_bf"]]
        + [("dtokens", c_vp), ("dx", c_vp * 2), ("dx16", c_vp * 2)]
        + [(n, c_vp) for n in ["dhid", "dxn", "d_o", "dqkv", "delta", "dacc", "attn_ws"]]
    )


EPI_BF16, EPI_GELU, EPI_RESID_F32, EPI_DGELU, EPI_F32, EPI_ATOMIC_F32, EPI_RESID_LN = range(7)

# name -> (restype, argtypes); mirrors include/mfvit.h one to one
SIGNATURES = {
    "mfv_abi_version": (C.c_int, []),
    "mfv_init": (C.c_int, [C.c_int]),
    "mfv_strerror": (C.c_char_p, [C.c_int]),
    "mfv_last_error_where": (C.c_char_p, []),
    "mfv_set_option": (C.c_int, [C.c_char_p, C.c_int]),
    "mfv_num_sms": (C.c_int, []),
    "mfv_launch_count": (C.c_uint64, []),
    "mfv_prof_enable": (C.c_int, [C.c_int]),
    "mfv_prof_num_labels": (C.c_int, []),
    "mfv_prof_label_name": (C.c_char_p, [C.c_int]),
    "mfv_prof_read": (C.c_int, [c_vp, c_vp, C.c_int]),
    "mfv_gemm": (C.c_int, [C.POINTER(GemmArgs), c_vp]),
    "mfv_gemm_wgrad_pair": (C.c_int, [C.POINTER(GemmArgs), C.POINTER(GemmArgs), c_vp]),
    "mfv_layernorm_fwd": (C.c_int, [c_vp, c_vp, c_vp, c_vp, C.c_int, c_vp, c_vp, c_vp, c_vp, i64, i64, i64, i64, f32, c_vp]),
    "mfv_layernorm_bwd": (C.c_int, [c_vp] * 13 + [i64, i64, i64, i64, c_vp]),
    "mfv_attn_fwd": (C.c_int, [c_vp, C.c_int, c_vp, C.c_int, c_vp, c_vp, i64, i64, i64, i64, f32, c_vp]),
    "mfv_attn_bwd": (C.c_int, [c_vp, C.c_int] + [c_vp] * 5 + [i64, i64, i64, i64, f32, c_vp]),
    "mfv_attn_bwd_workspace_bytes": (C.c_size_t, [i64, i64, i64, i64]),
    "mfv_attn_bwd_ws": (C.c_int, [c_vp, C.c_int] + [c_vp] * 6 + [i64, i64, i64, i64, f32, c_vp]),
    "mfv_attn_probs": (C.c_int, [c_vp, C.c_int, c_vp, c_vp, i64, i64, i64, i64, f32, c_vp]),
    "mfv_attn_rollout": (C.c_int, [c_vp, c_vp, i64, i64, i64, c_vp]),
    "mfv_patchify": (C.c_int, [c_vp, c_vp, C.c_int, c_vp, i64, i64, c_vp]),
    "mfv_debug_patch_tma_probe": (C.c_int, [c_vp, c_vp, i64, i64, i64, i64, i64, c_vp]),
    "mfv_patch_embed_tma": (C.c_int, [c_vp, c_vp, c_vp, C.c_int, c_vp, c_vp, c_vp, c_vp, i64, i64, i64, i64, i64, c_vp]),
    "mfv_embed_finish": (C.c_int, [c_vp] * 5 + [i64] * 5 + [c_vp]),
    "mfv_embed_finish_bwd": (C.c_int, [c_vp] * 4 + [i64] * 5 + [c_vp]),
    "mfv_colsum_bf16": (C.c_int, [c_vp, c_vp, i64, i64, i64, i64, c_vp]),
    "mfv_fusion_saved_floats": (C.c_size_t, [i64, i64, i64, i64]),
    "mfv_fusion_fwd": (C.c_int, [c_vp, C.POINTER(FusionParams), c_vp, c_vp, c_vp, i64, i64, i64, i64, i64, c_vp]),
    "mfv_fusion_bwd": (C.c_int, [c_vp, C.POINTER(FusionParams), c_vp, c_vp, c_vp, c_vp, C.POINTER(FusionGrads),
                                 i64, i64, i64, i64, i64, c_vp]),
    "mfv_fusion_bwd_deferred": (C.c_int, [c_vp, C.POINTER(FusionParams), c_vp, c_vp, c_vp, c_vp, C.POINTER(FusionGrads),
                                 i64, i64, i64, i64, i64, c_vp]),
    "mfv_fusion_bwd_join": (C.c_int, [c_vp]),
    "mfv_fusion_attn": (C.c_int, [c_vp, C.POINTER(FusionParams), c_vp, i64, i64, i64, i64, c_vp]),
    "mfv_linear_small_fwd": (C.c_int, [c_vp, i64, c_vp, c_vp, c_vp, i64, i64, i64, c_vp]),
    "mfv_linear_small_bwd": (C.c_int, [c_vp, i64, c_vp, c_vp, c_vp, i64, c_vp, c_vp, i64, i64, i64, c_vp]),
    "mfv_ce_small": (C.c_int, [c_vp] * 6 + [i64, i64, c_vp]),
    "mfv_augment_u8": (C.c_int, [c_vp] * 5 + [i64, i64, i64, i64, c_vp]),
    "mfv_epoch_metrics": (C.c_int, [c_vp] * 5 + [i64, i64, c_vp, c_vp, i64, c_vp, c_vp, c_vp, c_vp]),
    "mfv_ema_update": (C.c_int, [c_vp, i64, i64, f32, f32, c_vp]),
    "mfv_infonce_fwd": (C.c_int, [c_vp] * 8 + [i64, i64, i64, f32, c_vp]),
    "mfv_infonce_bwd": (C.c_int, [c_vp] * 8 + [i64, i64, f32, c_vp, i64, i64, i64, f32, c_vp]),
    "mfv_infonce_tc_fwd": (C.c_int, [c_vp] * 7 + [i64, c_vp, c_vp, i64, i64, i64, f32, c_vp]),
    "mfv_infonce_tc_bwd": (C.c_int, [c_vp] * 5 + [i64, c_vp, c_vp, c_vp, i64, i64, f32, c_vp, c_vp, c_vp, i64, i64, i64,
                                     f32, c_vp]),
    "mfv_queue16_update": (C.c_int, [c_vp, c_vp, i64, i64, i64, i64, c_vp]),
    "mfv_enqueue_keys": (C.c_int, [c_vp, c_vp, i64, i64, i64, i64, c_vp]),
    "mfv_vit_forward": (C.c_int, [C.POINTER(VitPlan), c_vp]),
    "mfv_vit_backward": (C.c_int, [C.POINTER(VitPlan), c_vp]),
    "mfv_vit_backward_range": (C.c_int, [C.POINTER(VitPlan), c_vp, C.c_int, C.c_int, C.c_int]),
    "mfv_cast_shadow": (C.c_int, [c_vp, c_vp, c_vp, i64, c_vp]),
    "mfv_cast_bf16_f32": (C.c_int, [c_vp, c_vp, i64, c_vp]),
    "mfv_fill_f32": (C.c_int, [c_vp, f32, i64, c_vp]),
    "mfv_sgd_step": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, i64, f32, f32, f32, C.c_int, c_vp]),
    "mfv_adam_step": (C.c_int, [c_vp] * 6 + [i64, f32, f32, f32, f32, f32, C.c_int, i64, c_vp]),
    "mfv_sgd_step_dev": (C.c_int, [c_vp, c_vp, c_vp, c_vp, c_vp, i64, c_vp, f32, f32, C.c_int, c_vp]),
    "mfv_adam_step_dev": (C.c_int, [c_vp] * 6 + [i64, c_vp, f32, f32, f32, f32, C.c_int, c_vp, c_vp]),
    "mfv_lars_workspace_bytes": (C.c_size_t, [i64]),
    "mfv_lars_step_dev": (C.c_int, [c_vp, i64, i64, c_vp, c_vp, c_vp, f32, f32, f32, c_vp]),
}

_lib = None
_lock = threading.Lock()
_inited_devices = set()


def load():
    """dlopen libmfvit.so and declare every prototype.  Works without a GPU (symbol check only)."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise MfvError(
                    "libmfvit.so not built (%s). Run `python multi-feature-vit_b200/build.py`; there is no fallback "
                    "path." % LIB_PATH)
            lib = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def check(rc, what="mfvit"):
    if rc != 0:
        msg = load().mfv_strerror(int(rc))
        where = load().mfv_last_error_where() if rc > 0 else b""
        raise MfvError("%s failed: %s (code %d)%s" % (what, msg.decode() if msg else "?", rc,
                                                       " at " + where.decode() if where else ""))


def init(device_index):
    """mfv_init on first use of a device (validates sm_100, resolves the TMA descriptor encoder)."""
    lib = load()
    if device_index not in _inited_devices:
        if _inited_devices:
            raise MfvError("libmfvit.so is bound to cuda:%d in this process; cuda:%d needs its own process (one process "
                           "per GPU: the side stream, events and kernel attributes are per-process state)"
                           % (next(iter(_inited_devices)), int(device_index)))
        check(lib.mfv_init(int(device_index)), "mfv_init")
        _inited_devices.add(device_index)
    return lib
