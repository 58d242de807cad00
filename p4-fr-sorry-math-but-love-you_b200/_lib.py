"""ctypes binding of include/frx.h (the reference-side stub a maintainer would
add; see INTEGRATION.md).  No torch types cross the boundary: tensors are
passed as raw device pointers and the current CUDA stream handle."""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None

SYMBOLS = [
    "frx_version", "frx_create", "frx_destroy", "frx_last_error", "frx_load_tensor",
    "frx_finalize_weights", "frx_encode", "frx_decode_greedy", "frx_forward_greedy",
    "frx_forward_greedy_host", "frx_forward_greedy_host_submit", "frx_forward_greedy_host_wait", "frx_decode_begin", "frx_decode_step", "frx_beam_search",
    "frx_decode_teacher_forced", "frx_launch_count", "frx_device_bytes", "frx_set_option",
    "frx_read_tap", "frx_last_timing", "frx_read_prof", "frx_tc_gemm",
    "frx_set_decoding_rules", "frx_decode_greedy_managed", "frx_forward_greedy_managed",
    "frx_train_create", "frx_train_destroy", "frx_train_param_count", "frx_train_fwd_bwd", "frx_train_grad_buffer",
    "frx_train_set_bucket_callback", "frx_train_apply", "frx_train_export", "frx_train_read_grad", "frx_train_step_count", "frx_train_read_tap",
    "frx_train_forward", "frx_train_backward", "frx_train_import", "frx_ensemble_decode", "frx_preprocess_u8", "frx_train_apply_dual",
    "frx_decode_greedy_eos", "frx_forward_greedy_eos", "frx_train_set_dropout", "frx_philox4x32",
]

BUCKET_CALLBACK = ctypes.CFUNCTYPE(None, ctypes.c_void_p, ctypes.c_int64, ctypes.c_int64)


class FrxConfig(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int32) for n in (
        "network", "height", "width", "in_ch",
        "enc_hidden", "enc_filter", "enc_layers", "enc_heads",
        "dec_src", "dec_hidden", "dec_filter", "dec_layers", "dec_heads",
        "num_classes", "sos_id", "eos_id", "pad_id",
        "max_batch", "max_steps", "precision", "device")]


def library_path() -> str:
    return os.environ.get("FRX_LIBRARY", os.path.join(_HERE, "lib", "libfrx.so"))


def load_library():
    """Load libfrx.so or fail loudly -- there is no fallback path."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = library_path()
    if not os.path.exists(path):
        raise RuntimeError(
            "frx: compiled CUDA library not found at %s. Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` (nvcc, sm_100a). "
            "There is no CPU/PyTorch fallback." % path)
    lib = ctypes.CDLL(path)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
    lib.frx_version.restype = ctypes.c_char_p
    lib.frx_last_error.restype = ctypes.c_char_p
    lib.frx_last_error.argtypes = [vp]
    lib.frx_create.argtypes = [ctypes.POINTER(FrxConfig), ctypes.POINTER(vp)]
    lib.frx_destroy.argtypes = [vp]
    lib.frx_destroy.restype = None
    lib.frx_load_tensor.argtypes = [vp, ctypes.c_char_p, vp, ctypes.POINTER(i64), i32, i32]
    lib.frx_finalize_weights.argtypes = [vp]
    lib.frx_forward_greedy_host_submit.argtypes = [vp, vp, i32, i32, vp, i32, vp]
    lib.frx_forward_greedy_host_wait.argtypes = [vp, i32]
    lib.frx_encode.argtypes = [vp, vp, i32, vp, vp]
    lib.frx_decode_greedy.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp]
    lib.frx_forward_greedy.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.frx_forward_greedy_host.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.frx_decode_begin.argtypes = [vp, vp, i32, vp]
    lib.frx_decode_step.argtypes = [vp, vp, vp, vp]
    lib.frx_beam_search.argtypes = [vp, vp, i32, i32, i32, vp, vp]
    lib.frx_decode_teacher_forced.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.frx_launch_count.argtypes = [vp]
    lib.frx_launch_count.restype = i64
    lib.frx_device_bytes.argtypes = [vp]
    lib.frx_device_bytes.restype = i64
    lib.frx_set_option.argtypes = [vp, ctypes.c_char_p, i64]
    lib.frx_read_tap.argtypes = [vp, ctypes.c_char_p, vp, i64, ctypes.POINTER(i64), ctypes.POINTER(i32), vp]
    lib.frx_read_prof.argtypes = [vp, ctypes.POINTER(i64)]
    lib.frx_tc_gemm.argtypes = [vp, vp, vp, vp, i32, i32, i32, ctypes.POINTER(i32), vp, vp, i32, i32, vp]
    lib.frx_last_timing.argtypes = [vp, ctypes.POINTER(ctypes.c_float)]
    lib.frx_set_decoding_rules.argtypes = [vp, ctypes.POINTER(i32), ctypes.POINTER(i32), i32, ctypes.POINTER(i32)]
    lib.frx_decode_greedy_managed.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.frx_forward_greedy_managed.argtypes = [vp, vp, i32, i32, vp, vp, vp]
    lib.frx_decode_greedy_eos.argtypes = [vp, vp, i32, i32, vp, vp, vp, vp, i32, vp]
    lib.frx_forward_greedy_eos.argtypes = [vp, vp, i32, i32, vp, vp, vp, i32, vp]
    f32 = ctypes.c_float
    lib.frx_train_create.argtypes = [vp, i32, i32, vp]
    lib.frx_train_destroy.argtypes = [vp]
    lib.frx_train_destroy.restype = None
    lib.frx_train_param_count.argtypes = [vp]
    lib.frx_train_param_count.restype = i64
    lib.frx_train_fwd_bwd.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.frx_train_grad_buffer.argtypes = [vp, ctypes.POINTER(vp), ctypes.POINTER(i64)]
    lib.frx_train_set_bucket_callback.argtypes = [vp, BUCKET_CALLBACK, vp]
    lib.frx_train_apply.argtypes = [vp, f32, f32, f32, f32, vp, vp]
    lib.frx_train_apply_dual.argtypes = [vp, f32, f32, f32, f32, f32, vp, vp, vp]
    lib.frx_train_export.argtypes = [vp, ctypes.c_char_p, vp]
    lib.frx_train_read_grad.argtypes = [vp, ctypes.c_char_p, vp]
    lib.frx_preprocess_u8.argtypes = [vp, ctypes.POINTER(i64), ctypes.POINTER(i32), ctypes.POINTER(i32), i32, i32, i32, i32,
                                      ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_float), i32, vp, vp]
    lib.frx_ensemble_decode.argtypes = [ctypes.POINTER(vp), i32, ctypes.POINTER(vp), i32, i32, vp, vp, i32, vp]
    lib.frx_train_forward.argtypes = [vp, vp, vp, i32, i32, vp, vp, vp]
    lib.frx_train_backward.argtypes = [vp, vp, vp, i32, i32, vp]
    lib.frx_train_import.argtypes = [vp, ctypes.c_char_p, vp]
    lib.frx_train_read_tap.argtypes = [vp, ctypes.c_char_p, vp, i64]
    lib.frx_train_read_tap.restype = i64
    lib.frx_train_step_count.argtypes = [vp]
    lib.frx_train_step_count.restype = i64
    lib.frx_train_set_dropout.argtypes = [vp, f32, f32, ctypes.c_uint64, i32]
    u32x = ctypes.POINTER(ctypes.c_uint32)
    lib.frx_philox4x32.argtypes = [u32x, u32x, u32x]
    _LIB = lib
    return lib


class Handle:
    """Owns one frx_handle*; every failing call raises RuntimeError with
    frx_last_error (the reference raises Python exceptions from torch)."""

    def __init__(self, cfg: FrxConfig):
        self.lib = load_library()
        self.ptr = ctypes.c_void_p()
        self.cfg = cfg
        rc = self.lib.frx_create(ctypes.byref(cfg), ctypes.byref(self.ptr))
        if rc != 0:
            msg = self.lib.frx_last_error(self.ptr).decode() if self.ptr else "frx_create failed"
            if self.ptr:
                self.lib.frx_destroy(self.ptr)
                self.ptr = ctypes.c_void_p()
            raise RuntimeError("frx_create: " + msg)

    def check(self, rc, what):
        if rc != 0:
            raise RuntimeError("%s: %s" % (what, self.lib.frx_last_error(self.ptr).decode()))

    def call(self, name, *args):
        self.check(getattr(self.lib, name)(self.ptr, *args), name)

    def close(self):
        if getattr(self, "ptr", None):
            self.lib.frx_destroy(self.ptr)
            self.ptr = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
