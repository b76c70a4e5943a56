"""Pin the oracle against (a) the reference's known-answer NMS vectors and (b) outputs of the
unmodified reference python captured in tests/golden/*.npz (generator: tests/golden/gen_golden.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import model as M
from oracle import ops as O
from oracle import postproc as P
from sipmask_b200 import synth


def _load(golden_dir, name):
    return dict(np.load(os.path.join(golden_dir, name)))


# ---- known-answer NMS (MM/tests/test_nms.py:17-41; nms_wrapper.py:25-34; BM/tests/test_nms.py:16-58)
def test_nms_mm_fixtures(golden_dir):
    g = _load(golden_dir, 'nms_known_answers.npz')
    for cmp_ge in (False, True):
        assert len(O.nms(g['mm4_dets'], float(g['mm4_thr']), cmp_ge=cmp_ge)) == int(g['mm4_num_keep'])
        assert len(O.nms(g['mm7_dets'], float(g['mm7_thr']), cmp_ge=cmp_ge)) == int(g['mm7_num_keep'])
    # the survey ran the reference's nms_cpu.cpp on the 4-box fixture: keep == [0, 2, 3]
    assert O.nms(g['mm4_dets'], 0.7, cmp_ge=True).tolist() == [0, 2, 3]


def _bm_boxlist(rows):
    """BM/tests/test_nms.py builds BoxList(..., mode='xywh').convert('xyxy'): x2 = x + w - 1 (TO_REMOVE = 1)."""
    b = np.asarray(rows, np.float32)
    return np.stack([b[:, 0], b[:, 1], b[:, 0] + b[:, 2] - 1, b[:, 1] + b[:, 3] - 1], 1)


def test_nms_bm_known_answers(golden_dir):
    """SipMask-benchmark/tests/test_nms.py:16-58 (5 boxes, five thresholds -> kept sets) and :60- (53 boxes ->
    gt_indices); the vectors are stored as data in nms_known_answers.npz by tests/golden/gen_golden.py."""
    g = _load(golden_dir, 'nms_known_answers.npz')
    dets5 = np.concatenate([g['bm5_boxes_xyxy'], g['bm5_scores'][:, None]], 1).astype(np.float32)
    for thr, want in zip(g['bm5_thrs'], g['bm5_keeps']):
        want = [int(i) for i in want if i >= 0]
        for cmp_ge in (False, True):
            assert sorted(O.nms(dets5, float(thr), cmp_ge=cmp_ge).tolist()) == sorted(want), (thr, cmp_ge)
    dets53 = np.concatenate([g['bm53_boxes_xyxy'], g['bm53_scores'][:, None]], 1).astype(np.float32)
    keep = O.nms(dets53, float(g['bm53_thr']), cmp_ge=True)
    assert sorted(keep.tolist()) == sorted(g['bm53_gt_indices'].tolist())


def nms_cpp_cases():
    """(key, dets [n,5] float32, iou threshold) of the comparison with the reference's nms_cpu.cpp."""
    rng = np.random.RandomState(0)
    for n in (1, 7, 64, 65, 300):
        xy = rng.rand(n, 2) * 200
        wh = rng.rand(n, 2) * 80 + 1
        dets = np.concatenate([xy, xy + wh, rng.rand(n, 1)], 1).astype(np.float32)
        for thr in (0.3, 0.5, 0.7):
            yield 'keep_%d_%g' % (n, thr), dets, thr


def test_nms_matches_reference_cpp(golden_dir):
    """oracle.ops.nms(cmp_ge=True) == what the reference's own nms_cpu.cpp kept on the same boxes (ref_nms_cpu.npz,
    generator: tests/golden/gen_golden_ref_native.py)."""
    g = _load(golden_dir, 'ref_nms_cpu.npz')
    for key, dets, thr in nms_cpp_cases():
        assert O.nms(dets, thr, cmp_ge=True).tolist() == g[key].tolist(), key


def test_c_oracle_matches_numpy():
    from oracle import cbind
    rng = np.random.RandomState(1)
    n = 200
    xy = rng.rand(n, 2) * 100
    wh = rng.rand(n, 2) * 60 + 1
    dets = np.concatenate([xy, xy + wh, rng.rand(n, 1)], 1).astype(np.float32)
    for cmp_ge in (0, 1):
        assert cbind.nms(dets, 0.5, cmp_ge).tolist() == O.nms(dets, 0.5, cmp_ge=bool(cmp_ge)).tolist()
    protos = torch.relu(torch.randn(32, 20, 28))
    cofs = torch.randn(5, 128)
    boxes = torch.tensor([[2.3, 1.2, 20.7, 15.1], [0, 0, 28, 20], [5, 5, 5.5, 5.5], [-3, -2, 9, 30], [10.5, 3.5, 11.5, 4.5]])
    pos, masks = P.assemble_masks(protos, cofs, boxes, torch.tensor([1.0]), 2.0, 0.4)
    c_pos = cbind.mask_assemble(protos.numpy(), cofs.numpy(), boxes.numpy())
    np.testing.assert_allclose(c_pos, pos.numpy(), atol=2e-6)
    stack = torch.rand(4, 20, 28, 5)
    np.testing.assert_array_equal(cbind.crop_split(stack.numpy(), (boxes * 0.5).numpy()), O.crop_split(stack, boxes * 0.5).numpy())
    c_masks = cbind.upsample2_thresh(c_pos, 0.4)
    assert (c_masks != masks.numpy()).mean() < 1e-3


# ---- reference python fixtures
@pytest.mark.parametrize('name,cmp_ge', [('ref_head_gn4.npz', True), ('ref_head_ssd2.npz', True),
                                         ('ref_head_gn4_sf.npz', True), ('ref_head_ssd2_sf.npz', True)])
def test_head_and_postproc_match_reference(golden_dir, name, cmp_ge):
    """The *_sf fixtures were produced with scale_factor != 1 and ori_shape != img_shape (rescale=True): boxes / scale_factor,
    masks interpolated by 2 / scale_factor (per axis on the SSD path) and pasted into the ori_shape canvas."""
    g = _load(golden_dir, name)
    stacked, gn, ssd = int(g['stacked_convs']), bool(g['gn']), bool(g['ssd_flag'])
    head = M.SipMaskHead(stacked_convs=stacked, gn=gn, ssd_flag=ssd)
    sd = synth.head_state_dict(seed=int(g['seed']), prefix='', stacked_convs=stacked, gn=gn, cls_bias=-2.0)
    head.load_state_dict(sd, strict=True)
    head.eval()
    nl = len(g['sizes'])
    feats = [torch.from_numpy(g['feat%d' % i]) for i in range(nl)]
    with torch.no_grad():
        cls, box, ctr, cof, fm = head(feats)
    for i in range(nl):
        np.testing.assert_allclose(cls[i].numpy(), g['cls%d' % i], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(box[i].numpy(), g['bbox%d' % i], rtol=1e-4, atol=1e-3)
        np.testing.assert_allclose(ctr[i].numpy(), g['ctr%d' % i], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(cof[i].numpy(), g['cof%d' % i], rtol=1e-4, atol=1e-4)
    np.testing.assert_allclose(fm.numpy(), g['feat_masks'], rtol=1e-4, atol=1e-4)

    # post-processing from the REFERENCE's head outputs -> must reproduce its detections exactly
    cfg = dict(nms_pre=int(g['nms_pre']), score_thr=float(g['score_thr']), nms=dict(iou_thr=0.5),
               max_per_img=int(g['max_per_img']))
    sf = g['scale_factor']
    sf = float(sf[0]) if sf.size == 1 else sf
    res = P.get_bboxes_single(
        [torch.from_numpy(g['cls%d' % i][0]) for i in range(nl)],
        [torch.from_numpy(g['bbox%d' % i][0]) for i in range(nl)],
        [torch.from_numpy(g['ctr%d' % i][0]) for i in range(nl)],
        [torch.from_numpy(g['cof%d' % i][0]) for i in range(nl)],
        torch.from_numpy(g['feat_masks'][0]), (8, 16, 32, 64, 128),
        tuple(g['img_shape']), tuple(g['ori_shape']), sf, cfg, rescale=True, ssd_flag=ssd, cmp_ge=cmp_ge)
    assert res['det_labels'].tolist() == g['det_labels'].tolist()
    np.testing.assert_array_equal(res['det_bboxes'].numpy(), g['det_bboxes'])
    assert res['masks'].shape == g['masks'].shape
    inter = np.logical_and(res['masks'], g['masks']).sum((1, 2))
    union = np.logical_or(res['masks'], g['masks']).sum((1, 2))
    assert ((inter + 1e-9) / (union + 1e-9)).min() >= 0.999
    assert (res['masks'] == g['masks']).all()


def rescore_fixture_inputs(g):
    """Regenerate the inputs of the compact ref_head_ssd2_rescore fixture (tests/golden/gen_golden.py::gen_head_case):
    seeded synthetic head weights incl. the rescoring layers, and the five feature maps from torch.Generator(seed + 10)."""
    seed = int(g['seed'])
    sd = synth.head_state_dict(seed=seed, prefix='', stacked_convs=int(g['stacked_convs']), gn=bool(g['gn']), cls_bias=-2.0,
                               rescoring_flag=True)
    gen = torch.Generator().manual_seed(seed + 10)
    feats = [torch.randn(1, 256, int(h), int(w), generator=gen) for (h, w) in g['sizes']]
    return sd, feats


def test_rescoring_matches_reference(golden_dir):
    """SipMask++ mask rescoring (sipmask_head.py:200-219,635-643) - fixture from the reference python run with
    rescoring_flag=True: the oracle must reproduce detections, masks and mask_scores."""
    g = _load(golden_dir, 'ref_head_ssd2_rescore.npz')
    sd, feats = rescore_fixture_inputs(g)
    head = M.SipMaskHead(stacked_convs=int(g['stacked_convs']), gn=bool(g['gn']), ssd_flag=True, rescoring_flag=True)
    head.load_state_dict(sd, strict=True)
    head.eval()
    with torch.no_grad():
        cls, box, ctr, cof, fm = head(feats)
        cfg = dict(nms_pre=int(g['nms_pre']), score_thr=float(g['score_thr']), nms=dict(iou_thr=0.5),
                   max_per_img=int(g['max_per_img']))
        res = P.get_bboxes_single([t[0] for t in cls], [t[0] for t in box], [t[0] for t in ctr], [t[0] for t in cof], fm[0],
                                  (8, 16, 32, 64, 128), tuple(g['img_shape']), tuple(g['ori_shape']), g['scale_factor'], cfg,
                                  rescale=True, ssd_flag=True, cmp_ge=True, head=head)
    assert res['det_labels'].tolist() == g['det_labels'].tolist()
    np.testing.assert_allclose(res['det_bboxes'].numpy(), g['det_bboxes'], rtol=1e-4, atol=1e-3)
    want = g['mask_scores']
    assert (want > 0).sum() >= 10                                     # the fixture exercises the non-trivial branch
    np.testing.assert_allclose(res['mask_scores'].numpy(), want, rtol=2e-3, atol=2e-5)
    ref_masks = np.unpackbits(g['masks'], axis=-1)[:, :, :int(g['mask_w'])]
    inter = np.logical_and(res['masks'], ref_masks).sum((1, 2))
    union = np.logical_or(res['masks'], ref_masks).sum((1, 2))
    assert ((inter + 1e-9) / (union + 1e-9)).min() >= 0.999


@pytest.mark.parametrize('name,depth,seed,dcn', [('ref_backbone_r50_64x96', 50, 1, (False,) * 4),
                                                 ('ref_backbone_r101_64x96', 101, 4, (False,) * 4),
                                                 ('ref_backbone_r50_dcn_64x96', 50, 6, (False, True, True, True))])
def test_backbone_fpn_match_reference(golden_dir, name, depth, seed, dcn):
    """Oracle ResNet + FPN vs the unmodified reference modules on the same weights / image: ResNet-50, ResNet-101 (config 3)
    and the `++` backbone with DeformConvPack in stages 2-4 (block 0 and every third block, resnet.py:288-291; the
    reference's DCN native call is bound to oracle.ops.deform_conv, which tests/test_gpu_ref_cuda.py pins against the
    reference CUDA kernel)."""
    g = _load(golden_dir, name + '.npz')
    net = M.ResNet(depth, dcn)
    net.load_state_dict(synth.backbone_state_dict(depth, seed, prefix='', stage_with_dcn=dcn), strict=True)
    fpn = M.FPN()
    fpn.load_state_dict(synth.neck_state_dict(seed + 1, prefix=''), strict=True)
    net.eval(), fpn.eval()
    with torch.no_grad():
        c = net(torch.from_numpy(g['img']))
        p = fpn(c)
    for i, t in enumerate(c):
        np.testing.assert_allclose(t[0, :8].numpy(), g['c%d_slice' % i], rtol=1e-4, atol=1e-4)
        np.testing.assert_allclose(t.double().abs().sum().item(), g['c%d_sum' % i][1], rtol=1e-5)
    for i, t in enumerate(p):
        np.testing.assert_allclose(t[0, :16].numpy(), g['p%d' % i], rtol=1e-4, atol=1e-4)


def test_deform_conv_matches_torchvision():
    """Cross-check of the DCN restatement (no reference vector exists): torchvision's deform_conv2d
    uses the same offset layout [dg, 2*k*k (dh,dw interleaved), H, W]."""
    from torchvision.ops import deform_conv2d
    g = torch.Generator().manual_seed(0)
    x = torch.randn(2, 16, 9, 11, generator=g)
    w = torch.randn(8, 16, 3, 3, generator=g)
    off = torch.randn(2, 4 * 18, 9, 11, generator=g) * 2.5
    a = O.deform_conv(x, off, w, 1, 1, 1, 4)
    b = deform_conv2d(x, off, w, padding=1)
    np.testing.assert_allclose(a.numpy(), b.numpy(), rtol=1e-4, atol=1e-4)
    # tiny input (smaller than the kernel) is zero-padded first (deform_conv.py:242-254)
    x = torch.randn(1, 8, 2, 2, generator=g)
    off = torch.randn(1, 18, 2, 2, generator=g)
    w = torch.randn(4, 8, 3, 3, generator=g)
    assert O.deform_conv(x, off, w, 1, 1, 1, 1).shape == (1, 4, 2, 2)


def test_rle_roundtrip():
    rng = np.random.RandomState(0)
    m = (rng.rand(13, 17) > 0.6).astype(np.uint8)
    counts = O.rle_counts(m)
    assert sum(counts) == m.size
    flat = np.concatenate([np.full(c, i % 2, np.uint8) for i, c in enumerate(counts)])
    assert (flat.reshape(17, 13).T == m).all()
    assert isinstance(O.rle_to_string(counts), bytes)
