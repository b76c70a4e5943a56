"""Pins for the two CUDA-only reference operators, against what the reference's OWN kernels computed.

`tests/golden/ref_cuda_kernels.npz` holds the outputs of `CropSplitKernelForward` / its backward
(MM/mmdet/ops/crop/src/crop_split_cuda_kernel.cu:19-163), the CropSplitGt kernels (crop_split_gt_cuda_kernel.cu:19-140) and
`deformable_im2col_gpu_kernel` (MM/mmdet/ops/dcn/src/deform_conv_cuda_kernel.cu:84-277), compiled for sm_100a from the
reference sources (recipe: oracle/build.py::build_ref_cuda; wrappers oracle/ref_cuda/*.cu) and run on the seeded inputs
built below (generator: tests/golden/gen_golden_ref_native.py).  Each test compares three things on those inputs:
    reference kernel (stored)  ==  oracle restatement (oracle/ops.py)  ==  smb kernel through the C ABI
which removes the circularity of tests/golden/gen_golden.py (there the reference python's two native calls are bound to
the oracle, because neither has a CPU build).

The full outputs are too large to commit, so each is stored as:
  * bit-exact comparisons: the SHA-256 of the whole output (-0.0 counted as 0.0, as assert_array_equal / torch.equal do)
    plus the values at fixed sample positions, which locate a difference;
  * comparisons with a tolerance: the zero pattern of the whole output (bit-packed), the values at SAMPLE fixed positions
    among its non-zeros, and its sum, absolute sum and absolute maximum.
"""
import hashlib
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

GOLDEN = 'ref_cuda_kernels.npz'
SAMPLE = 4096                # stored values of an output compared with a tolerance
EXACT_SAMPLE = 1024          # stored values of an output compared bit for bit (the digest covers the rest)


# ---------------------------------------------------------------------------------------------------- inputs
def _rois(N, H, W, g):
    cx, cy = torch.rand(N, generator=g) * W, torch.rand(N, generator=g) * H
    bw, bh = torch.rand(N, generator=g) * W * 0.8 + 0.3, torch.rand(N, generator=g) * H * 0.8 + 0.3
    r = torch.stack([cx - bw / 2, cy - bh / 2, cx + bw / 2, cy + bh / 2], 1)
    fixed = torch.tensor([[0, 0, W, H], [-5, -7, W + 9, H + 3], [3.2, 4.1, 30.7, 35.2], [10, 10, 10.5, 10.5],
                          [0.5, 0.5, 1.5, 1.5], [20, 20, 19, 19], [W - 1, H - 1, W, H], [7, 3, 8, H - 1],
                          [4, 4, 12, 12], [4.0, 4.0, 11.9, 11.9]], dtype=torch.float32)
    r[:fixed.shape[0]] = fixed[:N]
    return r.contiguous()


def crop_split_inputs(H, W, N):
    """data [4,H,W,N] strictly positive (zeros mark "outside the box"), rois [N,4]; CPU fp32."""
    g = torch.Generator().manual_seed(H * 7 + N)
    data = torch.rand(4, H, W, N, generator=g) + 0.01
    return data, _rois(N, H, W, g)


def mask_assembly_inputs(H, W, N, sf):
    """protos [32,H,W], cofs [N,128], image-space boxes [N,4] (rois = boxes * sf / 2); CPU fp32."""
    from sipmask_b200 import synth
    g = torch.Generator().manual_seed(N)
    protos = synth.prototypes(H, W, seed=N)
    cofs = torch.randn(N, 128, generator=g)
    return protos, cofs, _rois(N, H, W, g) * 2.0 / sf


def deform_inputs(B, C, H, W, dg):
    """x [B,C,H,W] fp16-representable (the smb path stores fp16), offsets [B,dg*18,H,W] with integer sampling points,
    points on the map's edge and rows far outside the map (the `h_im > -1` predicate); CPU fp32."""
    g = torch.Generator().manual_seed(C + H)
    x = torch.randn(B, C, H, W, generator=g).half().float()
    off = torch.randn(B, dg * 18, H, W, generator=g) * 2.5
    off[:, :, 0, 0] = 0.0
    off[:, :, -1, -1] = torch.round(off[:, :, -1, -1])
    off[:, 0::2, 1, :] = -3.7
    return x, off


DEFORM_CONV_SHAPE = (1, 256, 25, 42, 4, 256)      # B, C, H, W, dg, Cout


def deform_conv_inputs():
    """x [B,C,H,W], offsets [B,dg*18,H,W], weight [Cout,C,3,3] (fp16-representable); CPU fp32."""
    B, C, H, W, dg, Cout = DEFORM_CONV_SHAPE
    g = torch.Generator().manual_seed(5)
    x = torch.randn(B, C, H, W, generator=g).half().float()
    off = torch.randn(B, dg * 18, H, W, generator=g) * 2.0
    weight = (torch.randn(Cout, C, 3, 3, generator=g) / 48.0).half().float()
    return x, off, weight


def crop_split_train_inputs(H, W, N):
    """rois, the gradient `top` [H,W,N], CropSplit input `data` [4,H,W,N] and CropSplitGt input `d` [H,W,N]; CPU fp32."""
    g = torch.Generator().manual_seed(H + N)
    rois = _rois(N, H, W, g)
    top = torch.rand(H, W, N, generator=g) + 0.01
    data = torch.rand(4, H, W, N, generator=g) + 0.01
    d = torch.rand(H, W, N, generator=g) + 0.01
    return rois, top, data, d


CROP_SPLIT_CASES = [(40, 56, 16), (100, 168, 37), (272, 272, 100)]
MASK_CASES = [(100, 168, 40, 1.0), (136, 136, 100, 1.0), (75, 125, 33, 1.6666)]
DEFORM_CASES = [(1, 256, 13, 21, 4), (2, 256, 25, 42, 4), (1, 128, 17, 17, 1), (1, 64, 7, 11, 1)]
TRAIN_CASES = [(40, 56, 16), (100, 168, 37)]


def case_key(name, *shape):
    return '%s_%s' % (name, '_'.join(str(s) for s in shape))


# --------------------------------------------------------------------------------------------- stored form
def sample_index(n, k):
    """k fixed positions in [0, n), ascending (all of them when n <= k)."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def _canonical(a):
    return np.ascontiguousarray(np.asarray(a, np.float32)).ravel() + np.float32(0)    # -0.0 + 0.0 = 0.0


def exact_entry(key, a):
    """What is stored of an output that must be reproduced bit for bit."""
    flat = _canonical(a)
    return {key + '__shape': np.asarray(a.shape, np.int64), key + '__sha256': np.asarray(hashlib.sha256(flat.tobytes()).hexdigest()),
            key + '__sample': flat[sample_index(flat.size, EXACT_SAMPLE)]}


def close_entry(key, a):
    """What is stored of an output that is compared with a tolerance (values kept in the output's dtype)."""
    a = np.asarray(a)
    flat = a.ravel()
    nz = np.flatnonzero(flat)
    return {key + '__shape': np.asarray(a.shape, np.int64), key + '__zeros': np.packbits(flat == 0),
            key + '__values': flat[nz[sample_index(nz.size, SAMPLE)]],
            key + '__sum': np.float64(flat.sum(dtype=np.float64)), key + '__abssum': np.float64(np.abs(flat).sum(dtype=np.float64)),
            key + '__absmax': np.float64(np.abs(flat).max())}


@pytest.fixture(scope='module')
def golden(golden_dir):
    return dict(np.load(os.path.join(golden_dir, GOLDEN)))


def assert_bits(got, golden, key):
    """got reproduces the stored reference output bit for bit."""
    got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else got
    assert list(got.shape) == golden[key + '__shape'].tolist(), (got.shape, key)
    flat = _canonical(got)
    np.testing.assert_array_equal(flat[sample_index(flat.size, EXACT_SAMPLE)], golden[key + '__sample'], err_msg=key)
    assert hashlib.sha256(flat.tobytes()).hexdigest() == str(golden[key + '__sha256']), key


class Stored(object):
    """A reference output compared with a tolerance: its zero pattern, sampled non-zeros and whole-array moments."""

    def __init__(self, golden, key):
        self.shape = tuple(golden[key + '__shape'].tolist())
        self.n = int(np.prod(self.shape))
        self.zero = np.unpackbits(golden[key + '__zeros'], count=self.n).astype(bool)
        nz = np.flatnonzero(~self.zero)
        self.idx = nz[sample_index(nz.size, SAMPLE)]
        self.values = golden[key + '__values']
        self.sum, self.abssum, self.absmax = (float(golden[key + s]) for s in ('__sum', '__abssum', '__absmax'))

    def flat(self, got):
        got = got.detach().cpu().numpy() if isinstance(got, torch.Tensor) else np.asarray(got)
        assert got.shape == self.shape, (got.shape, self.shape)
        return got.ravel()

    def assert_close(self, got, atol, rtol):
        """|got - ref| <= atol + rtol |ref| at the stored positions, and the sum of got within the bound that the same
        inequality at every element implies."""
        np.testing.assert_allclose(got[self.idx], self.values, atol=atol, rtol=rtol)
        assert abs(got.sum(dtype=np.float64) - self.sum) <= atol * self.n + rtol * self.abssum, (got.sum(dtype=np.float64), self.sum)


# --------------------------------------------------------------------------------------------------- tests
@pytest.mark.parametrize('H,W,N', CROP_SPLIT_CASES)
def test_crop_split_reference_kernel_vs_oracle_vs_smb(golden, H, W, N):
    from oracle import ops as O
    from sipmask_b200 import ops
    data, rois = crop_split_inputs(H, W, N)
    key = case_key('crop_split', H, W, N)
    assert_bits(O.crop_split(data, rois, 2), golden, key)                    # the restatement IS the reference kernel, bit for bit
    assert_bits(ops.crop_split(data.cuda(), rois.cuda()), golden, key)       # and so is the drop-in operator


@pytest.mark.parametrize('H,W,N,sf', MASK_CASES)
def test_mask_assembly_vs_reference_pipeline(golden, H, W, N, sf):
    """sipmask_head.py:615-627 with the reference's own CropSplit kernel:  4x (P @ cof_k^T) -> sigmoid -> stack ->
    CropSplitKernelForward -> permute, all fp32 on the GPU, versus the fused smb_mask_assemble.  The pipeline is also
    recomputed in full with the oracle's CropSplit (bit for bit the reference kernel, test above) and pinned to the stored
    output, so that every element of the smb output is compared."""
    from oracle import ops as O
    from sipmask_b200 import ops
    protos, cofs, boxes = mask_assembly_inputs(H, W, N, sf)
    ref = Stored(golden, case_key('mask_assembly', H, W, N, sf))
    P, cofs_d, boxes_d = protos.cuda().permute(1, 2, 0).contiguous(), cofs.cuda(), boxes.cuda()
    maps = torch.stack([torch.sigmoid(P @ cofs_d[:, 32 * k:32 * k + 32].t()) for k in range(4)], 0)     # [4,H,W,N]
    pipe = ref.flat(O.crop_split(maps.cpu(), (boxes_d * (sf / 2.0)).cpu(), 2).permute(2, 0, 1))
    assert ((pipe == 0) == ref.zero).all()
    ref.assert_close(pipe, atol=1e-6, rtol=0)                                # the same fp32 GEMM + sigmoid on the same device
    got = ref.flat(ops.mask_assemble(protos.cuda(), cofs_d, boxes_d, sf / 2.0, layout='chw'))
    assert ((got == 0) == ref.zero).all()                                    # crop + cell geometry identical to the reference kernel
    ref.assert_close(got, atol=5e-6, rtol=0)                                 # 32-term fp32 dot + sigmoid: summation order only
    np.testing.assert_allclose(got, pipe, atol=5e-6, rtol=0)


@pytest.mark.parametrize('B,C,H,W,dg', DEFORM_CASES)
def test_deformable_im2col_reference_kernel_vs_oracle_vs_smb(golden, B, C, H, W, dg):
    from oracle import ops as O
    from sipmask_b200 import conv
    x, off = deform_inputs(B, C, H, W, dg)
    ref = Stored(golden, case_key('deform_im2col', B, C, H, W, dg))         # [B, C*9, HW], row = c*9 + tap
    orc, _, _ = O.deform_im2col(x, off, 3, 3, 1, 1, 1, dg)
    orc = ref.flat(orc)
    # identical predicates / gather indices; the reference is compiled with FMA contraction, torch CPU is not
    ref.assert_close(orc, atol=2e-6, rtol=1e-6)
    assert ((orc == 0) == ref.zero).mean() > 0.9999
    # smb kernel: NHWC fp16 in, [N,H,W,tap*C + c] fp16 out
    col = conv.deform_im2col(x.permute(0, 2, 3, 1).contiguous().half().cuda(), off.permute(0, 2, 3, 1).contiguous().cuda(), dg)
    col = ref.flat(col.float().cpu().view(B, H * W, 9, C).permute(0, 3, 2, 1).reshape(B, C * 9, H * W))
    tol = 2e-3 * (ref.absmax + 1.0)                                          # one fp16 rounding of the output
    ref.assert_close(col, atol=tol, rtol=0)
    # every element, against the restatement: the same bound widened by the restatement's distance to the reference
    assert np.abs(col - orc).max() <= tol + 2e-6 + 1e-6 * ref.absmax


def test_deform_conv_operator_vs_reference_im2col_gemm(golden):
    """ops.DeformConv (drop-in for mmdet.ops.DeformConv, dcn/deform_conv.py:192-255) against the reference's
    im2col kernel followed by the weight GEMM (deform_conv_cuda.cpp:231-236), fp32 on the GPU.  Every element is also
    compared with the oracle's im2col followed by an fp64 GEMM, within the same bound widened by how far that product can
    lie from the reference's (|weight| times the im2col tolerance of the test above)."""
    from oracle import ops as O
    from sipmask_b200 import ops
    B, C, H, W, dg, Cout = DEFORM_CONV_SHAPE
    x, off, weight = deform_conv_inputs()
    m = ops.DeformConv(C, Cout, 3, stride=1, padding=1, deformable_groups=dg).cuda()
    with torch.no_grad():
        m.weight.copy_(weight)
    want = Stored(golden, case_key('deform_conv', *DEFORM_CONV_SHAPE))
    got = m(x.cuda(), off.cuda())
    assert got.shape == (B, Cout, H, W) and got.dtype == x.dtype
    got = want.flat(got.double())
    tol = 4e-3 * (want.absmax + 1.0)                                         # fp16 column + fp16 output, fp32 accumulate
    want.assert_close(got, atol=tol, rtol=0)
    col, _, _ = O.deform_im2col(x, off, 3, 3, 1, 1, 1, dg)                   # [B, C*9, HW]
    w = weight.view(Cout, C * 9).double()
    orc = want.flat((w @ col[0].double()).view(B, Cout, H, W))
    slack = (w.abs() @ (2e-6 + 1e-6 * col[0].double().abs())).max().item()
    want.assert_close(orc, atol=slack, rtol=0)
    assert np.abs(got - orc).max() <= tol + slack


@pytest.mark.parametrize('H,W,N', TRAIN_CASES)
def test_crop_split_backward_and_gt_vs_reference_kernels(golden, H, W, N):
    """Training-side companions (SURVEY 8f-4): CropSplit backward and CropSplitGt forward / backward against the reference's
    own kernels (crop_split_cuda_kernel.cu:90-163, crop_split_gt_cuda_kernel.cu:19-140), bit for bit, incl. autograd."""
    from sipmask_b200 import ops
    rois, top, data, d = (t.cuda() for t in crop_split_train_inputs(H, W, N))
    key = case_key('crop_split_backward', H, W, N)
    assert_bits(ops.crop_split_backward(top, rois), golden, key)
    data.requires_grad_(True)
    ops.CropSplit(2)(data, rois).backward(top)
    assert_bits(data.grad, golden, key)
    # CropSplitGt
    assert_bits(ops.CropSplitGt(2)(d, rois), golden, case_key('crop_split_gt', H, W, N))
    dg = d.clone().requires_grad_(True)
    ops.CropSplitGt(2)(dg, rois).backward(top)
    assert_bits(dg.grad, golden, case_key('crop_split_gt_backward', H, W, N))
