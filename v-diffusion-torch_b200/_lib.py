"""ctypes binding of the C ABI (include/vdt_b200.h) + the in-tree build of the CUDA library.

There is deliberately no fallback: if the shared library is missing or fails to load, every entry
point raises.  PyTorch is used only for device memory and streams; no torch type crosses the ABI.
"""
import ctypes as C
import glob
import os
import shutil
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(PKG_DIR, "csrc")
LIB_DIR = os.path.join(PKG_DIR, "lib")
LIB_PATH = os.environ.get("VDT_LIB", os.path.join(LIB_DIR, "libvdt_b200.so"))   # VDT_LIB: A/B-test another build
INCLUDE = os.path.join(os.path.dirname(PKG_DIR), "include", "vdt_b200.h")

VDT_MAX_LEVELS = 8
OUT_TYPES = {"x0": 0, "eps": 1, "both": 2, "v": 3}
VAR_TYPES = {"fixed_small": 0, "fixed_large": 1, "fixed_medium": 2}
SCHEDULES = {"cosine": 0, "linear": 1, "sigmoid": 2, "legacy": 3}
COEF_STRIDE = 16
OPERAND_DTYPES = {"fp16": 0, "bf16": 1, "fp16x3": 2}
REWEIGHT_TYPES = {"constant": 0, "snr": 1, "snr_trunc": 2, "snr_1plus": 3}
SOLVERS = {None: 0, "dpmpp_2m": 1}                # include/vdt_b200.h VDT_SOLVER_*


class UNetConfig(C.Structure):
    _fields_ = [("in_channels", C.c_int32), ("hid_channels", C.c_int32), ("out_channels", C.c_int32),
                ("num_levels", C.c_int32), ("ch_multipliers", C.c_int32 * VDT_MAX_LEVELS),
                ("num_res_blocks", C.c_int32), ("apply_attn", C.c_int32 * VDT_MAX_LEVELS),
                ("embedding_dim", C.c_int32), ("head_dim", C.c_int32), ("num_heads", C.c_int32),
                ("num_classes", C.c_int32), ("multitags", C.c_int32), ("resolution", C.c_int32),
                ("max_rows", C.c_int32), ("operand_dtype", C.c_int32)]


class SamplerConfig(C.Structure):
    _fields_ = [("sample_timesteps", C.c_int32), ("model_out_type", C.c_int32), ("model_var_type", C.c_int32),
                ("logsnr_schedule", C.c_int32), ("use_ddim", C.c_int32), ("x0eps_coef", C.c_int32),
                ("t_fp32", C.c_int32), ("solver", C.c_int32), ("intp_frac", C.c_double), ("logsnr_min", C.c_double), ("logsnr_max", C.c_double),
                ("w_guide", C.c_double), ("seed", C.c_uint64)]


class Inpaint(C.Structure):                               # include/vdt_b200.h vdt_inpaint
    _fields_ = [("known", C.c_void_p), ("mask", C.c_void_p), ("known_noise", C.c_void_p)]


class ConvOp(C.Structure):                                # include/vdt_b200.h vdt_conv_op
    _fields_ = [("a3", C.c_void_p), ("a3_lo", C.c_void_p), ("a1", C.c_void_p), ("a1_lo", C.c_void_p),
                ("w3", C.c_void_p), ("w1", C.c_void_p), ("bias", C.c_void_p), ("residual", C.c_void_p),
                ("out_f32", C.c_void_p), ("out16", C.c_void_p), ("stats", C.c_void_p), ("sat_count", C.c_void_p),
                ("batch", C.c_int32), ("h", C.c_int32), ("w", C.c_int32), ("c3", C.c_int32), ("c1", C.c_int32),
                ("cout", C.c_int32), ("ups", C.c_int32), ("resid_mode", C.c_int32), ("stat_cols", C.c_int32),
                ("f16", C.c_int32)]


def nvcc_path():
    for cand in (os.environ.get("NVCC"), shutil.which("nvcc"), "/usr/local/cuda/bin/nvcc"):
        if cand and os.path.exists(cand):
            return cand
    raise RuntimeError("nvcc not found (set NVCC)")


def sources():
    return sorted(glob.glob(os.path.join(CSRC, "*.cu")))


def needs_build():
    if not os.path.exists(LIB_PATH):
        return True
    t = os.path.getmtime(LIB_PATH)
    deps = sources() + glob.glob(os.path.join(CSRC, "*.cuh")) + [INCLUDE]
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """Compile every CUDA source for sm_100a into lib/libvdt_b200.so (in-tree, so it travels with
    the repo snapshot to the GPU box)."""
    if not force and not needs_build():
        return LIB_PATH
    os.makedirs(LIB_DIR, exist_ok=True)
    cmd = [nvcc_path(), "-shared", "-Xcompiler", "-fPIC", "-gencode", "arch=compute_100a,code=sm_100a", "-O3",
           "-lineinfo", "-std=c++17", "-o", LIB_PATH] + sources()
    if verbose:
        print(" ".join(cmd))
    subprocess.run(cmd, check=True)
    return LIB_PATH


_lib = None


def lib():
    """Load the library (never builds implicitly on a GPU box without nvcc; raises if absent)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU or PyTorch fallback for this path)")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.vdt_last_error.restype = C.c_char_p
    L.vdt_version.restype = C.c_int
    L.vdt_kernel_launches.restype = C.c_uint64
    L.vdt_plan_create.argtypes = [C.POINTER(UNetConfig), C.POINTER(vp)]
    L.vdt_plan_destroy.argtypes = [vp]
    L.vdt_plan_destroy.restype = None
    L.vdt_plan_num_weights.argtypes = [vp]
    L.vdt_plan_weight_name.argtypes = [vp, C.c_int]
    L.vdt_plan_weight_name.restype = C.c_char_p
    L.vdt_plan_weight_shape.argtypes = [vp, C.c_int, C.POINTER(i64), C.POINTER(C.c_int)]
    L.vdt_plan_load_weight.argtypes = [vp, C.c_char_p, vp, i64, C.c_int]
    L.vdt_plan_finalize.argtypes = [vp]
    L.vdt_unet_forward.argtypes = [vp, vp, vp, vp, vp, i32, vp]
    L.vdt_p_sample.argtypes = [vp, C.POINTER(SamplerConfig), vp, vp, vp, vp, i32, vp]
    L.vdt_p_sample_range.argtypes = [vp, C.POINTER(SamplerConfig), vp, vp, vp, i32, i32, i32, vp, vp]
    L.vdt_p_sample_inpaint.argtypes = [vp, C.POINTER(SamplerConfig), C.POINTER(Inpaint), vp, vp, vp, vp, i32, vp]
    L.vdt_p_sample_range_inpaint.argtypes = [vp, C.POINTER(SamplerConfig), C.POINTER(Inpaint), vp, vp, vp, i32, i32, i32, vp, vp]
    L.vdt_p_sample_from.argtypes = [vp, C.POINTER(SamplerConfig), C.POINTER(Inpaint), vp, vp, vp, i32, i32, vp]
    L.vdt_ddim_invert_range.argtypes = [vp, C.POINTER(SamplerConfig), vp, vp, i32, i32, i32, vp]
    L.vdt_invert_coefficients.argtypes = [C.POINTER(SamplerConfig), vp]
    L.vdt_op_invert_step.argtypes = [vp, vp, vp, i32, i32, i32, i32, i32, vp, C.c_float, vp]
    L.vdt_plan_flops.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_double)]
    L.vdt_profile_enable.argtypes = [C.c_int]
    L.vdt_profile_read.argtypes = [C.POINTER(C.c_double), C.POINTER(C.c_uint64)]
    L.vdt_p_sample_host.argtypes = [vp, C.POINTER(SamplerConfig), vp, vp, vp, vp, i32]
    L.vdt_step_coefficients.argtypes = [C.POINTER(SamplerConfig), vp]
    L.vdt_op_conv.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, vp, vp, vp, i32, vp, vp, i32, vp]
    L.vdt_op_conv_ex.argtypes = [C.POINTER(ConvOp), vp]
    L.vdt_op_in_conv.argtypes = [vp, i32, i32, i32, i32, i32, vp, vp, i32, vp, vp, i32, i32, vp]
    L.vdt_op_out_conv.argtypes = [vp, i32, i32, i32, i32, vp, i32, vp, vp, i32, vp]
    L.vdt_op_groupnorm.argtypes = [vp, i32, vp, i32, i32, i32, i32, vp, vp, vp, i32, i32, i32, i32, vp, vp, vp, i32, vp, vp, i32, i32, vp]
    L.vdt_op_attention.argtypes = [vp, vp, i32, i32, i32, i32, i32, vp]
    L.vdt_op_sampler_step.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, C.c_float, vp]
    L.vdt_op_sampler_step_hist.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, C.c_float, vp, vp]
    L.vdt_op_sampler_step_known.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, i32, i32, vp, C.c_float, vp, vp, vp, vp,
                                            C.c_uint64, vp, vp]
    L.vdt_stat_slabs_per_image.argtypes = [i32, i32]
    L.vdt_unet_forward_train.argtypes = [vp, vp, vp, vp, vp, i32, C.c_float, C.c_uint64, vp]
    L.vdt_op_groupnorm_dropout.argtypes = [vp, i32, i32, i32, i32, vp, vp, i32, vp, i32, C.c_float, C.c_uint64, i32, vp]
    L.vdt_plan_conv_flops_executed.argtypes = [vp, i32, vp]
    L.vdt_op_attention_backward.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    L.vdt_grad_sq_scratch_bytes.argtypes = [C.c_int64]
    L.vdt_grad_sq_scratch_bytes.restype = C.c_int64
    L.vdt_grad_sq_accumulate.argtypes = [vp, C.c_int64, vp, C.c_int64, vp, vp]
    L.vdt_adamw_ema_step.argtypes = [vp, vp, vp, vp, vp, C.c_int64, C.c_double, C.c_double, C.c_double, C.c_double, C.c_double, i32,
                                     vp, C.c_double, C.c_double, vp]
    L.vdt_op_groupnorm_backward.argtypes = [vp, vp, i32, i32, i32, i32, vp, vp, vp, i32, C.c_float, C.c_uint64, i32, vp, vp, vp, vp, vp]
    L.vdt_op_conv_dgrad.argtypes = [vp, i32, i32, i32, i32, vp, i32, i32, vp, i32, vp]
    L.vdt_op_conv_wgrad.argtypes = [vp, vp, i32, i32, i32, i32, i32, i32, vp, vp, i32, vp]
    L.vdt_train_coefficients.argtypes = [C.POINTER(SamplerConfig), vp, i32, vp]
    L.vdt_q_sample.argtypes = [vp, vp, vp, vp, i32, i32, vp]
    L.vdt_train_loss.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i32, i32, i32, i32, vp]
    L.vdt_images_to_uint8.argtypes = [vp, vp, i32, i32, i32, vp]
    L.vdt_plan_saturations.argtypes = [vp, C.POINTER(C.c_uint64), C.c_int]
    L.vdt_op_groupnorm_train.argtypes = [vp, i32, i32, i32, i32, vp, vp, vp, i32, i32, i32, vp, i32, C.c_float, C.c_uint64, i32, vp]
    L.vdt_op_linear.argtypes = [vp, vp, vp, vp, i32, i32, i32, i32, vp]
    L.vdt_op_timestep_embedding.argtypes = [vp, vp, i32, i32, vp]
    _lib = L
    return L


EXPORTS = ["vdt_last_error", "vdt_version", "vdt_kernel_launches", "vdt_plan_create", "vdt_plan_destroy",
           "vdt_plan_num_weights", "vdt_plan_weight_name", "vdt_plan_weight_shape", "vdt_plan_load_weight",
           "vdt_plan_finalize", "vdt_unet_forward", "vdt_p_sample", "vdt_p_sample_range", "vdt_p_sample_host",
           "vdt_p_sample_inpaint", "vdt_p_sample_range_inpaint", "vdt_p_sample_from", "vdt_ddim_invert_range",
           "vdt_invert_coefficients", "vdt_op_invert_step",
           "vdt_step_coefficients", "vdt_plan_flops", "vdt_profile_enable", "vdt_profile_read",
           "vdt_op_conv", "vdt_op_conv_ex", "vdt_op_in_conv", "vdt_op_out_conv", "vdt_op_groupnorm", "vdt_op_attention", "vdt_op_sampler_step", "vdt_op_sampler_step_hist",
           "vdt_op_sampler_step_known",           "vdt_stat_slabs_per_image",
           "vdt_plan_saturations", "vdt_images_to_uint8",
           "vdt_train_coefficients", "vdt_q_sample", "vdt_train_loss", "vdt_unet_forward_train", "vdt_op_groupnorm_dropout",
           "vdt_op_conv_dgrad", "vdt_op_conv_wgrad", "vdt_op_groupnorm_backward",
           "vdt_plan_conv_flops_executed", "vdt_grad_sq_scratch_bytes", "vdt_grad_sq_accumulate", "vdt_adamw_ema_step",
           "vdt_op_attention_backward", "vdt_op_groupnorm_train", "vdt_op_linear", "vdt_op_timestep_embedding"]


def check(rc):
    if rc != 0:
        raise RuntimeError("vdt_b200: " + lib().vdt_last_error().decode())


def ptr(t):
    """Device (or host) address of a contiguous torch tensor, None -> NULL."""
    if t is None:
        return None
    assert t.is_contiguous()
    return C.c_void_p(t.data_ptr())


def current_stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
