"""ctypes binding of libsnn_b200.so — the C-ABI declared in include/snnb.h.

There is no fallback: if the shared library is missing, `lib()` raises. (CPU-only hosts can still load it and
query symbols; any call that needs a device returns an error status with `snnb_last_error()` text.)
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "libsnn_b200.so")

c_float_p = C.POINTER(C.c_float)
c_int_p = C.POINTER(C.c_int)
vp = C.c_void_p


class ConvDesc(C.Structure):
    """snnb_conv_desc"""
    _fields_ = [
        ("in_channels", C.c_int),
        ("out_channels", C.c_int),
        ("kernel", C.c_int),
        ("stride", C.c_int),
        ("pad_x", C.c_int),
        ("pad_y", C.c_int),
        ("pad_mode", C.c_int),
        ("activation", C.c_int),
        ("leaky_alpha", C.c_float),
        ("algo", C.c_int),
    ]


class ModelOptions(C.Structure):
    """snnb_model_options"""
    _fields_ = [
        ("batch", C.c_int),
        ("input_width", C.c_int),
        ("input_height", C.c_int),
        ("conv_algo", C.c_int),
        ("use_cuda_graph", C.c_int),
        ("fuse", C.c_int),
        ("precision", C.c_int),
    ]


class ImageIO(C.Structure):
    """snnb_image_io"""
    _fields_ = [
        ("input_u8", C.c_void_p),
        ("src_height", C.c_int),
        ("src_width", C.c_int),
        ("linear_filter", C.c_int),
        ("mean4", C.c_float * 4),
        ("norm4", C.c_float * 4),
        ("output_f32", C.c_void_p),
        ("output_capacity", C.c_size_t),
        ("output_u8", C.c_void_p),
        ("out_scale", C.c_float),
        ("out_offset", C.c_float),
        ("classes_1based", C.c_void_p),
    ]


# name -> (restype, argtypes): every symbol include/snnb.h declares
SIGNATURES = {
    "snnb_version": (C.c_int, []),
    "snnb_last_error": (C.c_char_p, []),
    "snnb_context_create": (C.c_int, [C.c_int, C.POINTER(vp)]),
    "snnb_context_destroy": (C.c_int, [vp]),
    "snnb_sync": (C.c_int, [vp]),
    "snnb_context_stream": (vp, [vp]),
    "snnb_launch_count": (C.c_uint64, [vp]),
    "snnb_context_set_precision": (C.c_int, [vp, C.c_int]),
    "snnb_tensor_alloc": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]),
    "snnb_tensor_free": (C.c_int, [vp]),
    "snnb_tensor_dims": (C.c_int, [vp, c_int_p, c_int_p, c_int_p, c_int_p]),
    "snnb_tensor_upload_nhwc": (C.c_int, [vp, vp, vp]),
    "snnb_tensor_download_nhwc": (C.c_int, [vp, vp, vp]),
    "snnb_tensor_upload_c4hw4": (C.c_int, [vp, vp, vp]),
    "snnb_tensor_download_c4hw4": (C.c_int, [vp, vp, vp]),
    "snnb_tensor_dump": (C.c_int, [vp, vp, C.c_char_p]),
    "snnb_weights_pack_conv2d": (C.c_int, [vp, C.POINTER(ConvDesc), vp, vp, vp, vp, vp, vp, C.POINTER(vp)]),
    "snnb_weights_pack_depthwise": (C.c_int, [vp, C.POINTER(ConvDesc), vp, vp, vp, vp, vp, vp, C.POINTER(vp)]),
    "snnb_weights_pack_dense": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, C.POINTER(vp)]),
    "snnb_weights_pack_channels": (C.c_int, [vp, C.c_int, vp, vp, vp, vp, C.POINTER(vp)]),
    "snnb_weights_free": (C.c_int, [vp]),
    "snnb_conv2d_launch": (C.c_int, [vp, C.POINTER(ConvDesc), vp, vp, vp, vp]),
    "snnb_depthwise_launch": (C.c_int, [vp, C.POINTER(ConvDesc), vp, vp, vp]),
    "snnb_maxpool_launch": (C.c_int, [vp, C.c_int, C.c_int, vp, vp]),
    "snnb_avgpool_launch": (C.c_int, [vp, C.c_int, C.c_int, vp, vp]),
    "snnb_add_launch": (C.c_int, [vp, C.c_int, C.c_float, vp, vp, vp]),
    "snnb_batchnorm_launch": (C.c_int, [vp, vp, C.c_int, C.c_float, vp, vp]),
    "snnb_activation_launch": (C.c_int, [vp, C.c_int, C.c_float, vp, vp]),
    "snnb_dense_launch": (C.c_int, [vp, vp, C.c_int, C.c_float, vp, vp]),
    "snnb_softmax_launch": (C.c_int, [vp, vp, vp]),
    "snnb_argmax1": (C.c_int, [vp, vp, c_int_p]),
    "snnb_flatten_launch": (C.c_int, [vp, vp, vp]),
    "snnb_concat_launch": (C.c_int, [vp, vp, vp, vp]),
    "snnb_upsample_launch": (C.c_int, [vp, C.c_float, C.c_int, vp, vp]),
    "snnb_pad_launch": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp]),
    "snnb_instancenorm_launch": (C.c_int, [vp, vp, C.c_int, C.c_float, vp, vp]),
    "snnb_subpixel_launch": (C.c_int, [vp, C.c_int, vp, vp]),
    "snnb_timer_create": (C.c_int, [vp, C.POINTER(vp)]),
    "snnb_timer_start": (C.c_int, [vp]),
    "snnb_timer_stop": (C.c_int, [vp]),
    "snnb_timer_elapsed_ms": (C.c_int, [vp, c_float_p]),
    "snnb_timer_destroy": (C.c_int, [vp]),
    "snnb_model_load_json": (C.c_int, [vp, C.c_char_p, C.POINTER(ModelOptions), C.POINTER(vp)]),
    "snnb_model_destroy": (C.c_int, [vp]),
    "snnb_model_num_layers": (C.c_int, [vp]),
    "snnb_model_layer_info": (C.c_int, [vp, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int, c_int_p, c_int_p, c_int_p, c_int_p]),
    "snnb_model_num_inputs": (C.c_int, [vp]),
    "snnb_model_num_outputs": (C.c_int, [vp]),
    "snnb_model_input_dims": (C.c_int, [vp, C.c_int, c_int_p, c_int_p, c_int_p, c_int_p]),
    "snnb_model_output_dims": (C.c_int, [vp, C.c_int, c_int_p, c_int_p, c_int_p, c_int_p]),
    "snnb_model_run": (C.c_int, [vp, vp, vp, C.c_size_t, vp]),
    "snnb_graph_capture_begin": (C.c_int, [vp]),
    "snnb_graph_capture_end": (C.c_int, [vp, C.POINTER(C.c_void_p)]),
    "snnb_graph_launch": (C.c_int, [vp]),
    "snnb_graph_destroy": (C.c_int, [vp]),
    "snnb_model_submit": (C.c_int, [vp, vp, vp, C.c_size_t, vp, c_int_p]),
    "snnb_model_submit_u8": (C.c_int, [vp, vp, vp, vp, vp, C.c_size_t, vp, c_int_p]),
    "snnb_model_submit_image": (C.c_int, [vp, C.POINTER(ImageIO), c_int_p]),
    "snnb_model_wait": (C.c_int, [vp, C.c_int]),
    "snnb_model_set_input": (C.c_int, [vp, C.c_int, vp]),
    "snnb_model_forward": (C.c_int, [vp]),
    "snnb_model_get_output": (C.c_int, [vp, C.c_int, vp, C.c_size_t]),
    "snnb_model_layer_output": (C.c_int, [vp, C.c_int, vp, C.c_size_t]),
    "snnb_model_dump_outputs": (C.c_int, [vp, C.c_char_p]),
    "snnb_model_time_layers": (C.c_int, [vp, c_float_p, C.c_int]),
    "snnb_model_launches_per_forward": (C.c_int, [vp]),
    "snnb_model_layer_kernel": (C.c_int, [vp, C.c_int, C.c_char_p, C.c_int]),
    "snnb_model_get_boxes": (C.c_int, [vp, C.c_int, c_float_p, C.c_int, c_int_p]),
    "snnb_model_weight_arena": (C.c_int, [vp, C.POINTER(vp), C.POINTER(C.c_size_t)]),
    "snnb_nccl_unique_id": (C.c_int, [C.c_char_p]),
    "snnb_nccl_comm_create": (C.c_int, [vp, C.c_int, C.c_int, C.c_char_p, C.POINTER(vp)]),
    "snnb_nccl_comm_destroy": (C.c_int, [vp]),
    "snnb_bcast_weights": (C.c_int, [vp, vp, C.c_int]),
    "snnb_register_layer": (C.c_int, [C.c_char_p, vp, vp]),
    "snnb_unregister_layer": (C.c_int, [C.c_char_p]),
    "snnb_layer_json_number": (C.c_int, [vp, C.c_char_p, C.POINTER(C.c_double)]),
    "snnb_layer_json_string": (C.c_int, [vp, C.c_char_p, C.c_char_p, C.c_int]),
    "snnb_layer_json_numbers": (C.c_int, [vp, C.c_char_p, C.POINTER(C.POINTER(C.c_double)), C.POINTER(C.c_size_t)]),
    "snnb_tensor_planes": (C.c_int, [vp, C.POINTER(vp), C.POINTER(vp), c_int_p]),
    "snnb_debug_streamk_schedule": (C.c_int, [C.c_int, C.c_int, C.c_int, c_int_p, C.c_int]),
    "snnb_debug_feed_plan": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, c_int_p]),
    "snnb_debug_kblock_schedule": (C.c_int, [C.c_int] * 7 + [c_int_p, C.c_int]),
}

_lib = None


class SnnbError(RuntimeError):
    pass


def lib():
    """Load libsnn_b200.so (once) and attach the prototypes. Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SnnbError(
                "%s is missing — build it with `python -m shadernn_b200._build` (or __graft_entry__.build()). "
                "shadernn_b200 has no CPU or PyTorch fallback." % LIB_PATH)
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)  # AttributeError if a declared symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc, what=""):
    if rc != 0:
        msg = lib().snnb_last_error()
        raise SnnbError("%s failed (status %d): %s" % (what or "snnb call", rc, msg.decode("utf-8", "replace") if msg else "?"))
