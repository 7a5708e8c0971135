"""ctypes binding of libcdc_b200.so (include/cdc_b200.h).  No torch types cross this boundary:
only raw device pointers (tensor.data_ptr()), sizes and the CUDA stream handle."""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("CDC_LIB_PATH") or os.path.join(_HERE, "libcdc_b200.so")  # override: A/B builds in tools/

# every symbol include/cdc_b200.h declares (the drop-in boundary) ...
SYMBOLS = [
    "cdc_create", "cdc_destroy", "cdc_last_error", "cdc_abi_version", "cdc_act_dtype", "cdc_load_weights", "cdc_finalize_weights",
    "cdc_has_context_net", "cdc_set_schedule", "cdc_schedule_index", "cdc_schedule_coeffs", "cdc_set_sampler",
    "cdc_schedule_coeffs5", "cdc_film_size", "cdc_get_film", "cdc_bind_io", "cdc_set_cond", "cdc_get_cond", "cdc_set_latent",
    "cdc_set_x", "cdc_get_x", "cdc_get_x0", "cdc_denoise_step", "cdc_decode", "cdc_decode_host", "cdc_launches_per_step",
    "cdc_launches_context", "cdc_flops_per_step", "cdc_saturation_count", "cdc_quantize", "cdc_cdf_lookup",
    "cdc_has_codec", "cdc_encode_analysis", "cdc_hyper_encode", "cdc_hyper_decode",
    "cdc_rans_streams_per_channel", "cdc_rans_scratch_bytes", "cdc_rans_max_bytes", "cdc_rans_encode", "cdc_rans_decode",
]
# ... and include/cdc_b200_tools.h (tests / profiling / A-B; same library)
TOOLS_SYMBOLS = [
    "cdc_set_plan_option", "cdc_num_step_ops", "cdc_step_op_name", "cdc_step_op_flops", "cdc_step_op_bytes", "cdc_run_step_op",
    "cdc_profile_step", "cdc_profile_graph", "cdc_test_conv", "cdc_test_attention", "cdc_test_gn", "cdc_step_op_describe",
]
OPT_FUSE_APPLY, OPT_KF, OPT_KF_S2, OPT_KF_MIN_PIXELS, OPT_KF_RING = range(5)
OPK_MEMSET, OPK_CONV, OPK_GN_STATS, OPK_GN_APPLY, OPK_ATTENTION = range(5)  # cdc_op_kind


class CdcConfig(C.Structure):
    _fields_ = [("base", C.c_int32), ("mults", C.c_int32 * 4), ("groups", C.c_int32), ("heads", C.c_int32),
                ("head_dim", C.c_int32), ("temb", C.c_int32), ("T", C.c_int32), ("latent_ch", C.c_int32),
                ("gn_eps", C.c_float)]


class TensorDesc(C.Structure):
    _fields_ = [("p", C.c_void_p), ("C", C.c_int32), ("Cphys", C.c_int32), ("H", C.c_int32), ("W", C.c_int32)]


class StepOpDesc(C.Structure):
    """include/cdc_b200_tools.h cdc_step_op_desc"""
    _fields_ = [("kind", C.c_int32), ("weight", C.c_char * 64), ("res_weight", C.c_char * 64), ("in_gn", C.c_char * 64),
                ("film_off", C.c_int32), ("mode", C.c_int32), ("ksize", C.c_int32), ("epi", C.c_int32), ("silu", C.c_int32),
                ("kernel", C.c_int32), ("bn", C.c_int32), ("cpg", C.c_int32), ("ch", C.c_int32), ("staged", C.c_int32),
                ("xk16", C.c_int32), ("tr", C.c_int32), ("res1", C.c_int32), ("apply", C.c_int32),
                ("src", TensorDesc * 2), ("residual", TensorDesc), ("out", TensorDesc), ("res_out", TensorDesc),
                ("gn_in_acc", C.c_void_p), ("gn_out_acc", C.c_void_p), ("gn_slots", C.c_int32),
                ("x", C.c_void_p), ("x0_out", C.c_void_p), ("xpad", C.c_void_p)]


_libs = {}
VARIANTS = {"product": "libcdc_b200.so", "bf16": "libcdc_b200_bf16.so", "tools": "libcdc_b200_tools.so"}


def build(verbose=False, what="all"):
    """Compile the extension in-tree for sm_100a (nvcc cross-compiles without a GPU): the product library, the bf16
    variant the precision tests measure and the tools variant (csrc/build.sh)."""
    import subprocess
    script = os.path.join(_HERE, "csrc", "build.sh")
    r = subprocess.run(["bash", script, what], capture_output=True, text=True)
    if verbose or r.returncode:
        print(r.stdout + r.stderr)
    if r.returncode:
        raise RuntimeError("building libcdc_b200*.so failed:\n" + r.stdout + r.stderr)
    return LIB_PATH


def _bind(L):
    p, i32, i64, f32p, i32p = C.c_void_p, C.c_int, C.c_int64, C.c_void_p, C.c_void_p
    fp = C.POINTER(C.c_float)
    L.cdc_create.argtypes = [C.POINTER(CdcConfig), i32, C.POINTER(p)]
    L.cdc_destroy.argtypes = [p]
    L.cdc_destroy.restype = None
    L.cdc_last_error.argtypes = [p]
    L.cdc_last_error.restype = C.c_char_p
    L.cdc_load_weights.argtypes = [p, C.c_char_p, p, C.POINTER(i64), i32]
    L.cdc_finalize_weights.argtypes = [p]
    L.cdc_has_context_net.argtypes = [p]
    L.cdc_set_schedule.argtypes = [p, i32]
    L.cdc_schedule_index.argtypes = [p, i32]
    L.cdc_schedule_coeffs.argtypes = [p, i32, fp, fp]
    L.cdc_set_sampler.argtypes = [p, i32, C.c_float, C.c_uint64]
    L.cdc_schedule_coeffs5.argtypes = [p, i32, fp, fp, fp, fp, fp]
    L.cdc_film_size.argtypes = [p]
    L.cdc_get_film.argtypes = [p, f32p, p]
    L.cdc_bind_io.argtypes = [p, i32, i32, i32]
    L.cdc_set_cond.argtypes = [p, f32p, f32p, f32p, f32p, p]
    L.cdc_get_cond.argtypes = [p, f32p, f32p, f32p, f32p, p]
    L.cdc_set_latent.argtypes = [p, f32p, p]
    L.cdc_has_codec.argtypes = [p]
    L.cdc_encode_analysis.argtypes = [p, f32p, f32p, p]
    L.cdc_hyper_encode.argtypes = [p, f32p, f32p, p]
    L.cdc_hyper_decode.argtypes = [p, f32p, f32p, f32p, p]
    L.cdc_set_x.argtypes = [p, f32p, p]
    L.cdc_get_x.argtypes = [p, f32p, i32, p]
    L.cdc_get_x0.argtypes = [p, f32p, p]
    L.cdc_denoise_step.argtypes = [p, i32, p]
    L.cdc_decode.argtypes = [p, p]
    L.cdc_decode_host.argtypes = [p, f32p, f32p, f32p, p]
    L.cdc_launches_per_step.argtypes = [p]
    L.cdc_launches_context.argtypes = [p]
    L.cdc_flops_per_step.argtypes = [p]
    L.cdc_flops_per_step.restype = C.c_double
    L.cdc_saturation_count.argtypes = [p, C.POINTER(C.c_uint64), i32, p]
    L.cdc_quantize.argtypes = [f32p, f32p, i32p, f32p, i64, i64, i64, p]
    L.cdc_cdf_lookup.argtypes = [i32p, f32p, i32p, i32p, i32p, i32p, f32p, i32, i64, i32p, i32p, i32p, i32p, i32p,
                                 i64, p]
    L.cdc_rans_streams_per_channel.argtypes = [i64]
    L.cdc_rans_scratch_bytes.argtypes = [i64, i64, i32]
    L.cdc_rans_scratch_bytes.restype = i64
    L.cdc_rans_max_bytes.argtypes = [i64, i64, i32]
    L.cdc_rans_max_bytes.restype = i64
    L.cdc_rans_encode.argtypes = [p, p, p, p, p, p, i64, i64, i32, p, p, i64, p, p]
    L.cdc_rans_decode.argtypes = [p, i64, p, p, p, p, p, i32, i64, i64, i32, p, p, p, p]
    # tools header
    L.cdc_set_plan_option.argtypes = [p, i32, i32]
    L.cdc_num_step_ops.argtypes = [p]
    L.cdc_step_op_name.argtypes = [p, i32]
    L.cdc_step_op_name.restype = C.c_char_p
    L.cdc_step_op_flops.argtypes = [p, i32]
    L.cdc_step_op_flops.restype = C.c_double
    L.cdc_step_op_bytes.argtypes = [p, i32]
    L.cdc_step_op_bytes.restype = C.c_double
    L.cdc_run_step_op.argtypes = [p, i32, i32, p]
    L.cdc_step_op_describe.argtypes = [p, i32, C.POINTER(StepOpDesc)]
    L.cdc_profile_step.argtypes = [p, i32, i32, fp, p]
    L.cdc_profile_graph.argtypes = [p, i32, fp, fp, p]
    L.cdc_test_conv.argtypes = [i32, p, i32, p, i32, i32, i32, i32, f32p, f32p, i32, i32, i32, i32, p, p, p, p]
    L.cdc_test_attention.argtypes = [p, p, i32, i32, i32, p]
    L.cdc_test_gn.argtypes = [p, p, p, f32p, f32p, f32p, i32, i32, i32, i32, C.c_float, p]
    for s in SYMBOLS + TOOLS_SYMBOLS:
        getattr(L, s)  # raises AttributeError if the headers and the library disagree
    if hasattr(L, "cdc_debug_graph_skip"):  # tools build only
        L.cdc_debug_graph_skip.argtypes = [p, i32]
    return L


def lib(variant="product"):
    """Load a build of the shared library; fail loudly if it is missing (no fallback path exists).
    variant: "product" (default; CDC_LIB_PATH overrides the file), "bf16" or "tools"."""
    if variant in _libs:
        return _libs[variant]
    path = LIB_PATH if variant == "product" else os.path.join(_HERE, VARIANTS[variant])
    if not os.path.exists(path):
        raise RuntimeError(f"{path} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(cdc_b200 has no CPU or PyTorch fallback)")
    _libs[variant] = _bind(C.CDLL(path))
    return _libs[variant]


def check(ctx, rc, what, L=None):
    if rc != 0:
        msg = (L or lib()).cdc_last_error(ctx)
        raise RuntimeError(f"{what} failed ({rc}): {msg.decode() if msg else ''}")
