"""ctypes loader for libsipmask_b200.so (the C ABI declared in include/sipmask_b200.h).

There is NO fallback: if the library is missing or the device is not sm_100 every op raises.
"""
import ctypes
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SMB_LIB_PATH: an instrumented build of the same sources (tools/build_trace_lib.sh), for profiling tools only
LIB_PATH = os.environ.get('SMB_LIB_PATH') or os.path.join(HERE, 'lib', 'libsipmask_b200.so')

F32, F16 = 0, 1


class SmbError(RuntimeError):
    pass


class Level(ctypes.Structure):
    _fields_ = [('cls', ctypes.c_void_p), ('ctr', ctypes.c_void_p), ('box', ctypes.c_void_p),
                ('cls_pitch', ctypes.c_int), ('ctr_pitch', ctypes.c_int), ('box_pitch', ctypes.c_int),
                ('h', ctypes.c_int), ('w', ctypes.c_int), ('stride', ctypes.c_int),
                ('box_scale', ctypes.c_float), ('box_mul', ctypes.c_float)]


class ConvDesc(ctypes.Structure):
    _fields_ = [(n, ctypes.c_int) for n in (
        'N', 'H', 'W', 'Cin', 'Cout', 'kh', 'kw', 'stride', 'pad', 'relu', 'has_bias', 'has_residual',
        'residual_upsample', 'res_h', 'res_w', 'out_dtype', 'gn_stats', 'in_pitch', 'out_pitch')]


class ConvLevel(ctypes.Structure):
    _fields_ = [('inp', ctypes.c_void_p), ('out', ctypes.c_void_p), ('residual', ctypes.c_void_p),
                ('gn_stats', ctypes.c_void_p), ('H', ctypes.c_int), ('W', ctypes.c_int), ('res_h', ctypes.c_int),
                ('res_w', ctypes.c_int)]


_lib = None

# every symbol include/sipmask_b200.h declares (checked by tests/test_abi.py)
SYMBOLS = [
    'smb_last_error', 'smb_version', 'smb_check_device', 'smb_mask_assemble', 'smb_mask_upsample2_threshold', 'smb_mask_upsample2_threshold_pack', 'smb_mask_resize_threshold', 'smb_mask_resize_threshold_pack', 'smb_mask_assemble_pack', 'smb_mask_set_tensor_dot',
    'smb_crop_split_forward', 'smb_crop_split_backward', 'smb_crop_split_gt', 'smb_mask_rle_counts', 'smb_rle_to_string', 'smb_conv3x3s2_relu_f32', 'smb_mask_rescore', 'smb_nms', 'smb_decode_workspace_bytes', 'smb_decode_topk',
    'smb_multiclass_nms_workspace_bytes', 'smb_multiclass_nms', 'smb_fast_nms_workspace_bytes', 'smb_fast_nms',
    'smb_gather_rows_f32', 'smb_gather_det_inputs', 'smb_gather_track_feats', 'smb_track_step', 'smb_conv_plan_create', 'smb_conv_plan_create_multi', 'smb_conv_plan_destroy', 'smb_conv_plan_set_max_ctas', 'smb_conv_set_min_tiles',
    'smb_conv_plan_info', 'smb_conv_run',
    'smb_groupnorm_relu_apply', 'smb_groupnorm_stats', 'smb_deform_im2col', 'smb_offset_conv1x1', 'smb_groupnorm_relu_apply_multi', 'smb_offset_conv1x1_multi', 'smb_deform_im2col_multi', 'smb_maxpool3x3s2',
    'smb_upsample_bilinear', 'smb_image_to_nhwc8', 'smb_preprocess_u8', 'smb_stem_plan_create', 'smb_stem_plan_create_s2d', 'smb_image_to_s2d16', 'smb_preprocess_u8_s2d',
]


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise SmbError('%s not found: run `python -c "import __graft_entry__ as g; g.build()"` '
                           '(there is no CPU / PyTorch fallback)' % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        L.smb_last_error.restype = ctypes.c_char_p
        for n in ('smb_decode_workspace_bytes', 'smb_multiclass_nms_workspace_bytes', 'smb_fast_nms_workspace_bytes'):
            getattr(L, n).restype = ctypes.c_size_t
        L.smb_conv_plan_destroy.restype = None
        _lib = L
    return _lib


def check(rc, what=''):
    if rc != 0:
        raise SmbError('%s failed (%d): %s' % (what, rc, lib().smb_last_error().decode()))


def ptr(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)


def stream_ptr():
    """The CURRENT device's current stream.  Callers run under `device_guard` / `torch.cuda.device(tensor.device)`, so this
    is the stream of the device that owns the tensors (not of whatever device happened to be current)."""
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _find_device(objs):
    import torch
    for o in objs:
        if isinstance(o, torch.Tensor):
            if o.is_cuda:
                return o.device
        elif isinstance(o, (list, tuple)):
            d = _find_device(o)
            if d is not None:
                return d
    return None


def device_guard(fn):
    """Run `fn` with the CUDA device of its first CUDA tensor argument made current, so that the stream passed to the C ABI,
    the per-device kernel attributes and every launch belong to the tensors' device (multi-GPU processes, head.cuda(1))."""
    import functools

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        import torch
        dev = _find_device(args) or _find_device(tuple(kwargs.values()))
        if dev is None or dev.index is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)
    return wrapper


def f4(vals):
    return (ctypes.c_float * 4)(*[float(v) for v in vals])
