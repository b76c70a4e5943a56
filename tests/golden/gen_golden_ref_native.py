"""Generate tests/golden/ref_cuda_kernels.npz and tests/golden/ref_nms_cpu.npz by running the reference's own native
operators on the seeded inputs of tests/test_gpu_ref_cuda.py and tests/test_oracle_golden.py.

Needs a CUDA device and what oracle/build.py compiles from the reference sources into oracle/_ref/
(libsipmask_ref_cuda.so: the CropSplit, CropSplitGt and deformable im2col kernels; sipmask_ref_nms_cpu: nms_cpu.cpp):
    python tests/golden/gen_golden_ref_native.py [OUTDIR]          (default: tests/golden)
The stored form of each output (digest + sample, or zero pattern + sample + moments) is defined in tests/test_gpu_ref_cuda.py.
"""
import ctypes
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.join(ROOT, 'oracle', '_ref')
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import test_gpu_ref_cuda as T  # noqa: E402
import test_oracle_golden as TO  # noqa: E402

_lib = None


def _ref():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(os.path.join(REF, 'libsipmask_ref_cuda.so'))
    return _lib


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def ref_crop_split(data, rois):
    """data [4,H,W,N] fp32 cuda, rois [N,4] fp32 cuda -> [H,W,N] (zero-initialised like ops/crop/crop_split.py:22)."""
    _, H, W, N = data.shape
    out = torch.zeros((H, W, N), dtype=torch.float32, device=data.device)
    torch.cuda.synchronize()
    assert _ref().ref_crop_split_forward(_p(data), _p(rois), _p(out), H, W, 2, N) == 0
    return out


def ref_deform_im2col(x, offset, dg, k=3, pad=1, stride=1, dil=1):
    """x [B,C,H,W], offset [B,dg*2*k*k,Ho,Wo] fp32 cuda -> col [C*k*k, B, Ho, Wo] fp32 (deform_conv_cuda.cpp:231-236)."""
    B, C, H, W = x.shape
    Ho = (H + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    Wo = (W + 2 * pad - (dil * (k - 1) + 1)) // stride + 1
    col = torch.zeros((C * k * k, B, Ho, Wo), dtype=torch.float32, device=x.device)
    torch.cuda.synchronize()
    assert _ref().ref_deformable_im2col(_p(x), _p(offset), C, H, W, k, pad, stride, dil, B, dg, _p(col)) == 0
    return col


def ref_train_kernel(name, src, rois, H, W, N, shape):
    """CropSplit backward / CropSplitGt forward / backward into a zero-initialised output (crop_split.py:35)."""
    out = torch.zeros(shape, dtype=torch.float32, device='cuda')
    torch.cuda.synchronize()
    assert getattr(_ref(), name)(_p(src), _p(rois), _p(out), H, W, 2, N) == 0
    return out


def cuda_outputs():
    """key -> ('exact' | 'close', reference output as a numpy array)."""
    out = {}
    for H, W, N in T.CROP_SPLIT_CASES:
        data, rois = T.crop_split_inputs(H, W, N)
        out[T.case_key('crop_split', H, W, N)] = 'exact', ref_crop_split(data.cuda(), rois.cuda()).cpu().numpy()
    for H, W, N, sf in T.MASK_CASES:
        # sipmask_head.py:615-627: 4x (P @ cof_k^T) -> sigmoid -> stack -> CropSplitKernelForward -> permute, fp32 on the GPU
        protos, cofs, boxes = T.mask_assembly_inputs(H, W, N, sf)
        P = protos.cuda().permute(1, 2, 0).contiguous()
        cofs, boxes = cofs.cuda(), boxes.cuda()
        maps = torch.stack([torch.sigmoid(P @ cofs[:, 32 * k:32 * k + 32].t()) for k in range(4)], 0).contiguous()
        ref = ref_crop_split(maps, (boxes * (sf / 2.0)).contiguous()).permute(2, 0, 1).contiguous()
        out[T.case_key('mask_assembly', H, W, N, sf)] = 'close', ref.cpu().numpy()
    for B, C, H, W, dg in T.DEFORM_CASES:
        x, off = T.deform_inputs(B, C, H, W, dg)
        col = ref_deform_im2col(x.cuda(), off.cuda(), dg)                                  # [C*9, B, H, W]
        out[T.case_key('deform_im2col', B, C, H, W, dg)] = 'close', col.permute(1, 0, 2, 3).reshape(B, C * 9, H * W).cpu().numpy()
    B, C, H, W, dg, Cout = T.DEFORM_CONV_SHAPE
    x, off, weight = T.deform_conv_inputs()
    col = ref_deform_im2col(x.cuda(), off.cuda(), dg)
    want = (weight.cuda().view(Cout, -1).double() @ col.view(C * 9, -1).double()).view(Cout, B, H, W).permute(1, 0, 2, 3)
    out[T.case_key('deform_conv', *T.DEFORM_CONV_SHAPE)] = 'close', want.contiguous().cpu().numpy()
    for H, W, N in T.TRAIN_CASES:
        rois, top, _, d = (t.cuda() for t in T.crop_split_train_inputs(H, W, N))
        out[T.case_key('crop_split_backward', H, W, N)] = 'exact', ref_train_kernel(
            'ref_crop_split_backward', top, rois, H, W, N, (4, H, W, N)).cpu().numpy()
        out[T.case_key('crop_split_gt', H, W, N)] = 'exact', ref_train_kernel(
            'ref_crop_split_gt_forward', d, rois, H, W, N, (H, W, N)).cpu().numpy()
        out[T.case_key('crop_split_gt_backward', H, W, N)] = 'exact', ref_train_kernel(
            'ref_crop_split_gt_backward', top, rois, H, W, N, (H, W, N)).cpu().numpy()
    return out


def nms_outputs():
    sys.path.insert(0, REF)
    import sipmask_ref_nms_cpu as ref
    return {key: ref.nms(torch.from_numpy(dets), thr).numpy().astype(np.int64) for key, dets, thr in TO.nms_cpp_cases()}


def main(outdir):
    stored = {}
    for key, (kind, a) in cuda_outputs().items():
        stored.update(T.exact_entry(key, a) if kind == 'exact' else T.close_entry(key, a))
    np.savez_compressed(os.path.join(outdir, T.GOLDEN), **stored)
    np.savez_compressed(os.path.join(outdir, 'ref_nms_cpu.npz'), **nms_outputs())


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else HERE)
