"""ctypes binding of libnhans_b200.so (include/nhans_b200.h).  No CPU fallback: a missing library or a
machine without a B200 raises."""
from __future__ import annotations

import ctypes
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("NHANS_B200_LIB") or os.path.join(_HERE, "libnhans_b200.so")     # override: A/B builds

# every symbol include/nhans_b200.h declares (tests check the library exports each of them)
SYMBOLS = [
    "nhans_create", "nhans_destroy", "nhans_last_error", "nhans_load_weights", "nhans_normalise", "nhans_stft",
    "nhans_stft_f32", "nhans_eval_loss",
    "nhans_embed", "nhans_masknet", "nhans_istft", "nhans_output_offsets", "nhans_enhance_batch", "nhans_enhance_f32", "nhans_sync", "nhans_sync_previous",
    "nhans_upload", "nhans_run", "nhans_download", "nhans_postmix", "nhans_host_alloc", "nhans_host_free", "nhans_event_record",
    "nhans_event_elapsed_ms", "nhans_profile_enable", "nhans_profile_get", "nhans_profile_reset",
    "nhans_profile_get_layer", "nhans_plan_json",
    "nhans_debug_read_buffer", "nhans_debug_read_batch", "nhans_debug_timeline", "nhans_debug_layer_stats", "nhans_device_info",
    "nhans_stream_open", "nhans_stream_step", "nhans_stream_step_post", "nhans_stream_close", "nhans_stream_emit_len",
]


def build(verbose=False):
    """Compile the CUDA extension in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    if not verbose:
        cmd.append("-s")
    subprocess.check_call(cmd)


_lib = None


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise RuntimeError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                           "(there is no CPU fallback)" % SO_PATH)
    lib = ctypes.CDLL(SO_PATH)
    c = ctypes
    vp, i32, i64 = c.c_void_p, c.c_int, c.c_int64
    lib.nhans_last_error.restype = c.c_char_p
    lib.nhans_last_error.argtypes = [vp]
    lib.nhans_plan_json.restype = c.c_char_p
    lib.nhans_plan_json.argtypes = [vp, i32]
    lib.nhans_create.argtypes = [i32, i32, i32, i32, c.POINTER(vp)]
    lib.nhans_destroy.argtypes = [vp]
    lib.nhans_destroy.restype = None
    lib.nhans_load_weights.argtypes = [vp, vp, vp, vp, i32]
    lib.nhans_normalise.argtypes = [vp, vp, vp, i32, i32, vp, vp]
    lib.nhans_stft.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    lib.nhans_stft_f32.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    lib.nhans_eval_loss.argtypes = [vp, vp, vp, i64, vp]
    lib.nhans_embed.argtypes = [vp, vp, i32, vp]
    lib.nhans_masknet.argtypes = [vp, vp, vp, i32, vp, vp, vp]
    lib.nhans_istft.argtypes = [vp, vp, vp, vp, i32, vp, vp, vp, vp]
    lib.nhans_output_offsets.argtypes = [vp, i32, vp]
    lib.nhans_enhance_batch.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.nhans_upload.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp]
    lib.nhans_run.argtypes = [vp]
    lib.nhans_download.argtypes = [vp, vp, vp, vp]
    lib.nhans_postmix.argtypes = [vp, c.c_float, i32, vp, vp, vp, vp]
    lib.nhans_sync.argtypes = [vp]
    lib.nhans_enhance_f32.argtypes = [vp, vp, vp, i32, vp, vp, vp, vp, i32, vp, vp, vp]
    lib.nhans_sync_previous.argtypes = [vp]
    lib.nhans_host_alloc.argtypes = [i64, c.POINTER(vp)]
    lib.nhans_host_free.argtypes = [vp]
    lib.nhans_host_free.restype = None
    lib.nhans_event_record.argtypes = [vp, i32]
    lib.nhans_event_elapsed_ms.argtypes = [vp, i32, i32, c.POINTER(c.c_double)]
    lib.nhans_profile_enable.argtypes = [vp, i32]
    lib.nhans_profile_get.argtypes = [vp, i32, vp]
    lib.nhans_profile_reset.argtypes = [vp]
    lib.nhans_profile_get_layer.argtypes = [vp, i32, i32, vp]
    lib.nhans_debug_read_buffer.argtypes = [vp, i32, i32, vp, i64]
    lib.nhans_debug_read_batch.argtypes = [vp, i32, vp, i64]
    lib.nhans_debug_timeline.argtypes = [vp, vp, i32]
    lib.nhans_device_info.argtypes = [vp, c.POINTER(i32), c.POINTER(i32), c.POINTER(i32), c.POINTER(i64)]
    lib.nhans_stream_open.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp]
    lib.nhans_stream_step.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    lib.nhans_stream_step_post.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    lib.nhans_stream_close.argtypes = [vp, i32, vp]
    lib.nhans_stream_emit_len.argtypes = [i64, i64, i32, c.POINTER(i64)]
    _lib = lib
    return lib
