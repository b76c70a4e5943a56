"""Host side of the tcgen05 convolution engine: weight packing (BN folding, K-major fp16) and plan objects.

Reference modules replaced: nn.Conv2d (+ eval BatchNorm2d, bias, residual add, ReLU) in
MM/mmdet/models/backbones/resnet.py:203-239, MM/mmdet/models/necks/fpn.py:138-178,
MM/mmdet/ops/conv_module.py:124-132, MM/mmdet/models/anchor_heads/sipmask_head.py:241-287.
Activations are NHWC fp16 torch tensors; all compute happens in libsipmask_b200.so.
"""
import ctypes

import torch

from . import _lib as L


def pack_weight(w, bn=None, eps=1e-5, cout_pad=None, device=None):
    """[Cout,Cin,kh,kw] fp32 (+ eval BN (gamma,beta,mean,var)) -> ([Cout_pad, kh*kw*Cin] fp16 K-major, bias fp32|None).

    K index = (r*kw + s)*Cin + ci, matching the tap order of the TMA producer.  Frozen BN
    (resnet.py:514-521) folds to w *= gamma/sqrt(var+eps), bias = beta - mean*gamma/sqrt(var+eps)."""
    w = w.detach().float()
    cout, cin, kh, kw = w.shape
    bias = None
    if bn is not None:
        gamma, beta, mean, var = [t.detach().float() for t in bn]
        s = gamma / torch.sqrt(var + eps)
        w = w * s.view(-1, 1, 1, 1)
        bias = beta - mean * s
    wk = w.permute(0, 2, 3, 1).reshape(cout, kh * kw * cin)
    cp = cout_pad or ((cout + 15) // 16 * 16)
    if cp != cout:
        wk = torch.cat([wk, wk.new_zeros(cp - cout, wk.shape[1])], 0)
        if bias is not None:
            bias = torch.cat([bias, bias.new_zeros(cp - cout)])
    wk = wk.to(torch.float16).contiguous()
    if device is not None:
        wk = wk.to(device)
        bias = bias.to(device) if bias is not None else None
    return wk, bias


def pack_stem_weight(w, bn, eps=1e-5, device=None):
    """7x7 stem [64,3,7,7] -> [64, 7*64] : K = r*64 + s*8 + c (s<7, c<3 real, rest zero)."""
    gamma, beta, mean, var = [t.detach().float() for t in bn]
    s = gamma / torch.sqrt(var + eps)
    w = w.detach().float() * s.view(-1, 1, 1, 1)
    out = w.new_zeros(64, 7, 8, 8)
    out[:, :, :7, :3] = w.permute(0, 2, 3, 1)           # [co, r, s, c]
    wk = out.reshape(64, 448).to(torch.float16).contiguous()
    bias = (beta - mean * s).contiguous()
    if device is not None:
        wk, bias = wk.to(device), bias.to(device)
    return wk, bias


def pack_stem_weight_s2d(w, bn, eps=1e-5, device=None):
    """7x7 stem [64,3,7,7] -> [64, 4*64] for the space-to-depth stem: K = a*64 + b*16 + (dy*2+dx)*4 + c holds filter tap
    (r, s) = (2a+dy, 2b+dx), channel c (taps with r == 7 or s == 7 and c == 3 are zero)."""
    gamma, beta, mean, var = [t.detach().float() for t in bn]
    s = gamma / torch.sqrt(var + eps)
    w = w.detach().float() * s.view(-1, 1, 1, 1)
    w8 = w.new_zeros(64, 4, 8, 8)                        # [co, c(3->4), r(7->8), s(7->8)]
    w8[:, :3, :7, :7] = w
    # [co, c, a, dy, b, dx] -> [co, a, b, dy, dx, c]
    wk = w8.view(64, 4, 4, 2, 4, 2).permute(0, 2, 4, 3, 5, 1).reshape(64, 256).to(torch.float16).contiguous()
    bias = (beta - mean * s).contiguous()
    if device is not None:
        wk, bias = wk.to(device), bias.to(device)
    return wk, bias


# the fields of smb_conv_plan_info, in the order the library writes them
PLAN_INFO_FIELDS = ('n_tile', 'n_tiles_n', 'tiles_m', 'pair', 'cluster', 'grid', 'out_tma', 'res_tma', 'stage_slots',
                    'epi_split', 'small')


def set_min_tiles(n):
    """Planner knob for plans created afterwards (smb_conv_set_min_tiles); returns the previous value."""
    return int(L.lib().smb_conv_set_min_tiles(int(n)))


class ConvPlan(object):
    """One convolution bound to fixed input / weight / output buffers (TMA descriptors are baked at creation)."""

    def __init__(self, x, weight, out, k, stride=1, relu=False, bias=None, residual=None, residual_upsample=False,
                 gn_stats=None, cin=None, alpha=1.0):
        assert x.is_cuda and x.dtype == torch.float16 and x.dim() == 4 and x.stride(3) == 1
        N, H, W, _ = x.shape
        cin = cin if cin is not None else x.shape[3]
        in_pitch = x.stride(2)
        assert x.stride(1) == W * in_pitch and x.stride(0) == H * W * in_pitch
        cout = weight.shape[0]
        assert weight.shape[1] == k * k * cin and weight.dtype == torch.float16 and weight.is_contiguous()
        assert out.stride(3) == 1
        out_pitch = out.stride(2)
        d = L.ConvDesc()
        d.N, d.H, d.W, d.Cin, d.Cout = N, H, W, cin, cout
        d.kh = d.kw = k
        d.stride = stride
        d.pad = k // 2
        d.relu = int(relu)
        d.has_bias = int(bias is not None)
        d.has_residual = int(residual is not None)
        d.residual_upsample = int(residual_upsample)
        if residual is not None:
            d.res_h, d.res_w = residual.shape[1], residual.shape[2]
            assert residual.dtype == torch.float16 and residual.is_contiguous() and residual.shape[3] == cout
        d.out_dtype = L.F32 if out.dtype == torch.float32 else L.F16
        d.gn_stats = int(gn_stats is not None)
        d.in_pitch = in_pitch
        d.out_pitch = out_pitch
        self._keep = (x, weight, out, bias, residual, gn_stats)
        self.bias, self.residual, self.gn_stats, self.alpha = bias, residual, gn_stats, float(alpha)
        self.handle = ctypes.c_void_p()
        self.dev = x.device
        with torch.cuda.device(self.dev):
            L.check(L.lib().smb_conv_plan_create(ctypes.byref(d), L.ptr(x), L.ptr(weight), L.ptr(out),
                                                 ctypes.byref(self.handle)), 'smb_conv_plan_create')
        self.out = out

    def set_max_ctas(self, n):
        L.check(L.lib().smb_conv_plan_set_max_ctas(self.handle, int(n)), 'smb_conv_plan_set_max_ctas')
        return self

    def info(self):
        """What the planner chose for this plan (smb_conv_plan_info): tile shape, pair / cluster mode, grid, epilogue."""
        vals = (ctypes.c_int * len(PLAN_INFO_FIELDS))()
        rc = L.lib().smb_conv_plan_info(self.handle, vals, len(PLAN_INFO_FIELDS))
        if rc < 0:
            L.check(rc, 'smb_conv_plan_info')
        return dict(zip(PLAN_INFO_FIELDS, (int(v) for v in vals)))

    def run(self, stream=None):
        if self.dev.index != torch.cuda.current_device():        # launch on the plan's device and ITS current stream
            with torch.cuda.device(self.dev):
                return self.run(stream)
        L.check(L.lib().smb_conv_run(self.handle, L.ptr(self.bias), L.ptr(self.residual), L.ptr(self.gn_stats),
                                     ctypes.c_float(self.alpha), stream if stream is not None else L.stream_ptr()),
                'smb_conv_run')
        return self.out

    def __del__(self):
        try:
            if self.handle:
                L.lib().smb_conv_plan_destroy(self.handle)
                self.handle = None
        except Exception:
            pass


class ConvPlanMulti(ConvPlan):
    """One stride-1 convolution with shared weights over several feature-pyramid levels = ONE launch
    (the reference loops over levels in python, sipmask_head.py:250-271)."""

    def __init__(self, xs, weight, outs, k, relu=False, bias=None, gn_stats=None, alpha=1.0):
        nl = len(xs)
        N = xs[0].shape[0]
        cin = xs[0].shape[3]
        in_pitch = xs[0].stride(2)
        out_pitch = outs[0].stride(2)
        cout = weight.shape[0]
        assert weight.shape[1] == k * k * cin and weight.dtype == torch.float16 and weight.is_contiguous()
        lv = (L.ConvLevel * nl)()
        for i, (x, o) in enumerate(zip(xs, outs)):
            assert x.is_cuda and x.dtype == torch.float16 and x.stride(3) == 1 and x.stride(2) == in_pitch
            assert x.shape[0] == N and x.stride(1) == x.shape[2] * in_pitch and x.stride(0) == x.shape[1] * x.shape[2] * in_pitch
            assert o.stride(3) == 1 and o.stride(2) == out_pitch and o.dtype == outs[0].dtype
            st = gn_stats[i] if gn_stats is not None else None
            lv[i] = L.ConvLevel(x.data_ptr(), o.data_ptr(), 0, st.data_ptr() if st is not None else 0, x.shape[1], x.shape[2], 0, 0)
        d = L.ConvDesc()
        d.N, d.H, d.W, d.Cin, d.Cout = N, 0, 0, cin, cout
        d.kh = d.kw = k
        d.stride = 1
        d.pad = k // 2
        d.relu = int(relu)
        d.has_bias = int(bias is not None)
        d.has_residual = 0
        d.out_dtype = L.F32 if outs[0].dtype == torch.float32 else L.F16
        d.gn_stats = int(gn_stats is not None)
        d.in_pitch = in_pitch
        d.out_pitch = out_pitch
        self._keep = (xs, weight, outs, bias, gn_stats, lv)
        self.bias, self.residual, self.gn_stats, self.alpha = bias, None, None, float(alpha)
        self.handle = ctypes.c_void_p()
        self.dev = xs[0].device
        with torch.cuda.device(self.dev):
            L.check(L.lib().smb_conv_plan_create_multi(ctypes.byref(d), nl, lv, L.ptr(weight), ctypes.byref(self.handle)),
                    'smb_conv_plan_create_multi')
        self.out = outs


class StemPlan(ConvPlan):
    """7x7/2 stem + folded BN + ReLU (resnet.py:448-460) on the padded NHWC8 image [N,H+6,W+8,8] with weights [64,448]
    (pack_stem_weight), or - s2d=True - on the space-to-depth image [N,H/2+3,W/2+4,16] with weights [64,256]
    (pack_stem_weight_s2d): the same convolution with 43 % fewer operand bytes."""

    def __init__(self, img8, weight, bias, out, N, H, W, s2d=False):
        self._keep = (img8, weight, bias, out)
        self.bias, self.residual, self.gn_stats, self.alpha = bias, None, None, 1.0
        self.handle = ctypes.c_void_p()
        self.dev = img8.device
        assert tuple(img8.shape) == ((N, H // 2 + 3, W // 2 + 4, 16) if s2d else (N, H + 6, W + 8, 8)) and img8.is_contiguous()
        assert tuple(weight.shape) == (64, 256 if s2d else 448)
        with torch.cuda.device(self.dev):
            if s2d:
                L.check(L.lib().smb_stem_plan_create_s2d(N, H, W, L.ptr(img8), L.ptr(weight), L.ptr(out),
                                                         ctypes.byref(self.handle)), 'smb_stem_plan_create_s2d')
            else:
                L.check(L.lib().smb_stem_plan_create(N, H, W, L.ptr(img8), L.ptr(weight), L.ptr(out),
                                                     ctypes.byref(self.handle)), 'smb_stem_plan_create')
        self.out = out


# ------------------------------------------------------------------------------------- small wrappers
@L.device_guard
def image_to_nhwc8(img, out=None):
    N, _, H, W = img.shape
    if out is None:
        out = torch.empty((N, H + 6, W + 8, 8), dtype=torch.float16, device=img.device)
    L.check(L.lib().smb_image_to_nhwc8(L.ptr(img.contiguous()), L.ptr(out), N, H, W, L.stream_ptr()), 'smb_image_to_nhwc8')
    return out


@L.device_guard
def image_to_s2d16(img, out=None):
    """img [N,3,H,W] fp32 -> the stem's space-to-depth input [N, H/2+3, W/2+4, 16] fp16 (smb_image_to_s2d16)."""
    N, _, H, W = img.shape
    if out is None:
        out = torch.empty((N, H // 2 + 3, W // 2 + 4, 16), dtype=torch.float16, device=img.device)
    L.check(L.lib().smb_image_to_s2d16(L.ptr(img.contiguous()), L.ptr(out), N, H, W, L.stream_ptr()), 'smb_image_to_s2d16')
    return out


@L.device_guard
def preprocess_u8(src, resized_hw, out, mean):
    """uint8 BGR HWC CUDA image -> resized (cv2 INTER_LINEAR, bit-exact) - mean -> zero-padded fp16 stem input: `out` is
    either the NHWC8 buffer [1, H+6, W+8, 8] (smb_preprocess_u8) or the space-to-depth buffer [1, H/2+3, W/2+4, 16]
    (smb_preprocess_u8_s2d); the layout is taken from its shape."""
    assert src.is_cuda and src.dtype == torch.uint8 and src.dim() == 3 and src.shape[2] == 3 and src.stride(2) == 1 \
        and src.stride(1) == 3
    assert out.dtype == torch.float16 and out.is_contiguous() and out.shape[0] == 1 and out.shape[3] in (8, 16)
    m = (ctypes.c_float * 3)(*[float(v) for v in mean])
    if out.shape[3] == 16:
        H, W = 2 * (out.shape[1] - 3), 2 * (out.shape[2] - 4)
        L.check(L.lib().smb_preprocess_u8_s2d(L.ptr(src), int(src.shape[0]), int(src.shape[1]), int(src.stride(0)),
                                              int(resized_hw[0]), int(resized_hw[1]), m, L.ptr(out), H, W, L.stream_ptr()),
                'smb_preprocess_u8_s2d')
        return out
    H, W = out.shape[1] - 6, out.shape[2] - 8
    L.check(L.lib().smb_preprocess_u8(L.ptr(src), int(src.shape[0]), int(src.shape[1]), int(src.stride(0)), int(resized_hw[0]),
                                      int(resized_hw[1]), m, L.ptr(out), H, W, L.stream_ptr()), 'smb_preprocess_u8')
    return out


@L.device_guard
def maxpool3x3s2(x, out=None):
    N, H, W, C = x.shape
    Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    if out is None:
        out = torch.empty((N, Ho, Wo, C), dtype=torch.float16, device=x.device)
    L.check(L.lib().smb_maxpool3x3s2(L.ptr(x), L.ptr(out), N, H, W, C, L.stream_ptr()), 'smb_maxpool3x3s2')
    return out


@L.device_guard
def groupnorm_stats(x, stats=None):
    N, H, W, C = x.shape
    if stats is None:
        stats = torch.empty((N, 32, 2), dtype=torch.int64, device=x.device)
    L.check(L.lib().smb_groupnorm_stats(L.ptr(x), N, H * W, C, x.stride(2), L.ptr(stats), L.stream_ptr()),
            'smb_groupnorm_stats')
    return stats


@L.device_guard
def groupnorm_relu_apply(x, stats, gamma, beta, eps=1e-5, relu=True):
    N, H, W, C = x.shape
    L.check(L.lib().smb_groupnorm_relu_apply(L.ptr(x), N, H * W, C, x.stride(2), L.ptr(stats), L.ptr(gamma), L.ptr(beta),
                                             ctypes.c_float(eps), int(relu), L.stream_ptr()), 'smb_groupnorm_relu_apply')
    return x


@L.device_guard
def offset_conv1x1(bbox, scale, weight, out=None):
    """bbox [N,H,W,>=4] fp32 channel-last (pitch = stride(2)); weight [n_off,4] fp32 -> [N,H,W,n_off] fp32."""
    N, H, W, _ = bbox.shape
    n_off = weight.shape[0]
    if out is None:
        out = torch.empty((N, H, W, n_off), dtype=torch.float32, device=bbox.device)
    L.check(L.lib().smb_offset_conv1x1(L.ptr(bbox), bbox.stride(2), ctypes.c_float(scale), L.ptr(weight), n_off, L.ptr(out),
                                       ctypes.c_longlong(N * H * W), L.stream_ptr()), 'smb_offset_conv1x1')
    return out


@L.device_guard
def deform_im2col(x, offset, dg, out=None):
    """x [N,H,W,C] fp16, offset [N,H,W,dg*18] fp32 -> col [N,H,W,9*C] fp16."""
    N, H, W, C = x.shape
    assert x.is_contiguous()
    if out is None:
        out = torch.empty((N, H, W, 9 * C), dtype=torch.float16, device=x.device)
    L.check(L.lib().smb_deform_im2col(L.ptr(x), L.ptr(offset), offset.stride(2), L.ptr(out), N, H, W, C, int(dg),
                                      L.stream_ptr()), 'smb_deform_im2col')
    return out


@L.device_guard
def upsample_bilinear(x, factor, out=None, out_choff=0, relu=False):
    N, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, H * factor, W * factor, C), dtype=torch.float16, device=x.device)
    L.check(L.lib().smb_upsample_bilinear(L.ptr(x), x.stride(2), L.ptr(out), out.stride(2), int(out_choff), N, H, W, C,
                                          int(factor), out.shape[1], out.shape[2], int(relu), L.stream_ptr()),
            'smb_upsample_bilinear')
    return out


# ------------------------------------------------------------------------------------- multi-level wrappers
def _parr(ts):
    return (ctypes.c_void_p * len(ts))(*[t.data_ptr() for t in ts])


def _iarr(vals):
    return (ctypes.c_int * len(vals))(*[int(v) for v in vals])


@L.device_guard
def groupnorm_relu_apply_multi(xs, stats, gamma, beta, eps=1e-5, relu=True):
    N, _, _, C = xs[0].shape
    L.check(L.lib().smb_groupnorm_relu_apply_multi(len(xs), _parr(xs), _parr(stats), _iarr([x.shape[1] for x in xs]),
                                                   _iarr([x.shape[2] for x in xs]), N, C, xs[0].stride(2), L.ptr(gamma),
                                                   L.ptr(beta), ctypes.c_float(eps), int(relu), L.stream_ptr()),
            'smb_groupnorm_relu_apply_multi')
    return xs


@L.device_guard
def offset_conv1x1_multi(bboxes, scales, weight, offs):
    N = bboxes[0].shape[0]
    sc = (ctypes.c_float * len(scales))(*[float(v) for v in scales])
    L.check(L.lib().smb_offset_conv1x1_multi(len(bboxes), _parr(bboxes), bboxes[0].stride(2), sc, L.ptr(weight),
                                             weight.shape[0], _parr(offs), _iarr([b.shape[1] for b in bboxes]),
                                             _iarr([b.shape[2] for b in bboxes]), N, L.stream_ptr()),
            'smb_offset_conv1x1_multi')
    return offs


@L.device_guard
def deform_im2col_multi(xs, offs, dg, cols):
    N, _, _, C = xs[0].shape
    L.check(L.lib().smb_deform_im2col_multi(len(xs), _parr(xs), _parr(offs), offs[0].stride(2), _parr(cols),
                                            _iarr([x.shape[1] for x in xs]), _iarr([x.shape[2] for x in xs]), N, C, int(dg),
                                            L.stream_ptr()), 'smb_deform_im2col_multi')
    return cols
