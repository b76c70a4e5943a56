"""Drop-in boundary: the heads keep the reference's constructor / state_dict / method contract (CPU checks) and
reproduce the reference head on the golden fixtures (GPU)."""
import os

import numpy as np
import pytest
import torch

from sipmask_b200 import synth


def test_state_dict_contract_matches_reference_keys():
    """synth.head_state_dict was loaded strict=True into the unmodified reference SipMaskHead when the golden fixtures
    were generated (tests/golden/gen_golden.py); the drop-in head must accept exactly the same keys."""
    from sipmask_b200.head import FCOSHead, SipMaskHead
    h = SipMaskHead(num_classes=81, in_channels=256, stacked_convs=4, strides=[8, 16, 32, 64, 128])
    sd = synth.head_state_dict(seed=3, prefix='', stacked_convs=4, gn=True)
    r = h.load_state_dict(sd, strict=True)
    assert not r.missing_keys and not r.unexpected_keys
    h2 = SipMaskHead(num_classes=81, in_channels=256, stacked_convs=2, ssd_flag=True, norm_cfg=None, strides=[8, 16, 32, 64, 128])
    # the reference registers feat_align.norm even when norm_cfg is None (sipmask_head.py:40); it is simply unused
    sd2 = synth.head_state_dict(seed=5, prefix='', stacked_convs=2, gn=False)
    r2 = h2.load_state_dict(sd2, strict=True)
    assert not r2.missing_keys and not r2.unexpected_keys
    f = FCOSHead(num_classes=81, in_channels=256)
    keys = set(f.state_dict().keys())
    assert 'cls_convs.3.gn.weight' in keys and 'fcos_centerness.bias' in keys and 'scales.4.scale' in keys
    with pytest.raises(NotImplementedError):
        h.loss()


def test_rle_matches_oracle():
    from oracle import ops as O
    from sipmask_b200 import rle
    rng = np.random.RandomState(0)
    for shape in ((1, 1), (7, 5), (64, 33)):
        m = (rng.rand(*shape) > 0.5).astype(np.uint8)
        assert rle.counts(m).tolist() == O.rle_counts(m)
        assert rle.encode(m)['counts'] == O.rle_to_string(O.rle_counts(m))
        assert rle.encode(m)['size'] == list(shape)
    assert rle.counts(np.ones((2, 2), np.uint8)).tolist() == [0, 4]


def rle_decode(rle):
    """COCO RLE dict -> [H,W] uint8 (inverse of pycocotools rleToString / rleEncode: 5-bit groups, delta vs counts[i-2])."""
    s = rle['counts']
    s = s.decode('ascii') if isinstance(s, bytes) else s
    counts, p = [], 0
    while p < len(s):
        x, k, more = 0, 0, True
        while more:
            c = ord(s[p]) - 48
            x |= (c & 0x1f) << (5 * k)
            more = bool(c & 0x20)
            p += 1
            k += 1
            if not more and (c & 0x10):
                x |= -1 << (5 * k)
        if len(counts) > 2:
            x += counts[-2]
        counts.append(x)
    h, w = rle['size']
    flat = np.concatenate([np.full(c, i & 1, np.uint8) for i, c in enumerate(counts)]) if counts else np.zeros(0, np.uint8)
    assert flat.size == h * w, (flat.size, h, w)
    return flat.reshape(w, h).T


def test_rle_decode_inverts_oracle_encoder():
    from oracle import ops as O
    rng = np.random.RandomState(1)
    for shape in ((1, 1), (9, 4), (64, 33), (200, 301)):
        m = (rng.rand(*shape) > 0.7).astype(np.uint8)
        np.testing.assert_array_equal(rle_decode({'size': list(shape), 'counts': O.rle_to_string(O.rle_counts(m))}), m)


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['ref_head_gn4.npz', 'ref_head_ssd2.npz', 'ref_head_gn4_sf.npz', 'ref_head_ssd2_sf.npz'])
def test_dropin_head_reproduces_reference(golden_dir, name):
    from sipmask_b200.head import SipMaskHead
    g = dict(np.load(os.path.join(golden_dir, name)))
    stacked, gn, ssd = int(g['stacked_convs']), bool(g['gn']), bool(g['ssd_flag'])
    head = SipMaskHead(num_classes=81, in_channels=256, stacked_convs=stacked, ssd_flag=ssd, strides=[8, 16, 32, 64, 128],
                       norm_cfg=dict(type='GN', num_groups=32, requires_grad=True) if gn else None)
    head.load_state_dict(synth.head_state_dict(seed=int(g['seed']), prefix='', stacked_convs=stacked, gn=gn, cls_bias=-2.0),
                         strict=True)
    head = head.cuda().eval()
    nl = len(g['sizes'])
    feats = tuple(torch.from_numpy(g['feat%d' % i]).cuda() for i in range(nl))
    cls, box, ctr, cof, fm = head(feats)
    torch.cuda.synchronize()

    def rel(a, b):
        a, b = a.double().cpu().flatten(), torch.from_numpy(b).double().flatten()
        return ((a - b).norm() / (b.norm() + 1e-12)).item()
    for i in range(nl):
        assert cls[i].shape == g['cls%d' % i].shape and box[i].shape == g['bbox%d' % i].shape
        assert rel(cls[i], g['cls%d' % i]) < 2e-2, i
        assert rel(box[i], g['bbox%d' % i]) < 2e-2, i
        assert rel(cof[i], g['cof%d' % i]) < 3e-2, i
    assert rel(fm.float(), g['feat_masks']) < 2e-2
    # post-processing through the head API on the REFERENCE's head outputs -> the reference's detections
    class Cfg(dict):
        __getattr__ = dict.get
    cfg = Cfg(nms_pre=int(g['nms_pre']), score_thr=float(g['score_thr']), nms=Cfg(type='nms', iou_thr=0.5),
              max_per_img=int(g['max_per_img']))
    sf = g['scale_factor']
    meta = dict(img_shape=tuple(g['img_shape']), ori_shape=tuple(g['ori_shape']), scale_factor=float(sf[0]) if sf.size == 1 else sf)
    outs = ([torch.from_numpy(g['cls%d' % i]).cuda() for i in range(nl)], [torch.from_numpy(g['bbox%d' % i]).cuda() for i in range(nl)],
            [torch.from_numpy(g['ctr%d' % i]).cuda() for i in range(nl)], [torch.from_numpy(g['cof%d' % i]).cuda() for i in range(nl)],
            torch.from_numpy(g['feat_masks']).cuda())
    det_bboxes, det_labels, cls_segms = head.get_bboxes(*outs, [meta], cfg, rescale=True)[0]
    # the fixture comes from the reference's CPU path (nms_cpu `>=` comparator); the product uses the CUDA comparator `>`.
    # With these continuous random boxes no IoU equals the threshold exactly, so both give the same result.
    assert det_labels.cpu().tolist() == g['det_labels'].tolist()
    np.testing.assert_allclose(det_bboxes.cpu().numpy(), g['det_bboxes'], rtol=1e-6, atol=1e-6)
    assert len(cls_segms) == 80 and sum(len(c) for c in cls_segms) == len(g['det_labels'])
    # every RLE the drop-in returns decodes to the reference's mask of that detection (per class, in detection order)
    seen = [0] * 80
    for i, lab in enumerate(g['det_labels'].tolist()):
        rle = cls_segms[lab][seen[lab]]
        seen[lab] += 1
        assert rle['size'] == list(g['masks'][i].shape)
        m, r = rle_decode(rle).astype(bool), g['masks'][i].astype(bool)
        iou = (np.logical_and(m, r).sum() + 1e-9) / (np.logical_or(m, r).sum() + 1e-9)
        assert iou >= 0.999, (i, iou)


@pytest.mark.gpu
def test_dropin_head_rescoring_reproduces_reference(golden_dir):
    """rescoring_flag=True: get_bboxes returns (cls_segms, mask_scores) like sipmask_head.py:659-660; compared with the
    reference python's own run (ref_head_ssd2_rescore.npz).  Head outputs come from the oracle head (fp32), so that this
    test isolates the post-processing + rescoring chain."""
    from oracle import model as M
    from sipmask_b200.head import SipMaskHead
    from test_oracle_golden import rescore_fixture_inputs
    g = dict(np.load(os.path.join(golden_dir, 'ref_head_ssd2_rescore.npz')))
    sd, feats = rescore_fixture_inputs(g)
    ohead = M.SipMaskHead(stacked_convs=int(g['stacked_convs']), gn=False, ssd_flag=True, rescoring_flag=True)
    ohead.load_state_dict(sd, strict=True)
    ohead.eval()
    with torch.no_grad():
        outs = ohead(feats)
    head = SipMaskHead(num_classes=81, in_channels=256, stacked_convs=int(g['stacked_convs']), ssd_flag=True, rescoring_flag=True,
                       strides=[8, 16, 32, 64, 128], norm_cfg=None)
    head.load_state_dict(sd, strict=True)
    head = head.cuda().eval()

    class Cfg(dict):
        __getattr__ = dict.get
    cfg = Cfg(nms_pre=int(g['nms_pre']), score_thr=float(g['score_thr']), nms=Cfg(type='nms', iou_thr=0.5),
              max_per_img=int(g['max_per_img']))
    meta = dict(img_shape=tuple(g['img_shape']), ori_shape=tuple(g['ori_shape']), scale_factor=g['scale_factor'])
    dev = [[t.cuda() for t in lst] for lst in outs[:4]] + [outs[4].cuda()]
    det_bboxes, det_labels, (cls_segms, mask_scores) = head.get_bboxes(*dev, [meta], cfg, rescale=True)[0]
    assert det_labels.cpu().tolist() == g['det_labels'].tolist()
    np.testing.assert_allclose(det_bboxes.cpu().numpy(), g['det_bboxes'], rtol=1e-4, atol=1e-3)
    labels = g['det_labels']
    for c in range(80):
        np.testing.assert_allclose(mask_scores[c], g['mask_scores'][labels == c], rtol=2e-3, atol=2e-5)
    ref_masks = np.unpackbits(g['masks'], axis=-1)[:, :, :int(g['mask_w'])]
    seen = [0] * 80
    for i, lab in enumerate(labels.tolist()):
        m, r = rle_decode(cls_segms[lab][seen[lab]]).astype(bool), ref_masks[i].astype(bool)
        seen[lab] += 1
        assert (np.logical_and(m, r).sum() + 1e-9) / (np.logical_or(m, r).sum() + 1e-9) >= 0.999, i


@pytest.mark.gpu
def test_dropin_head_batch_and_engine_cache():
    """ADVICE r1: a batched forward must not crash (images are looped), outputs must not alias engine buffers, and a second
    resolution must not evict / repack the first one's engine or the shared packed weights."""
    from sipmask_b200.head import SipMaskHead
    head = SipMaskHead(num_classes=81, in_channels=256, stacked_convs=4, strides=[8, 16, 32, 64, 128])
    head.load_state_dict(synth.head_state_dict(seed=3, prefix='', stacked_convs=4, gn=True, cls_bias=-2.0), strict=True)
    head = head.cuda().eval()
    g = torch.Generator().manual_seed(0)
    sizes = [(12, 16), (6, 8), (3, 4), (2, 2), (1, 1)]
    f2 = tuple(torch.randn(2, 256, h, w, generator=g).cuda() for h, w in sizes)
    out2 = head(f2)
    eng_a = head._engine(f2)
    wcache = head._wcache
    single = [head(tuple(f[i:i + 1] for f in f2)) for i in range(2)]
    for i in range(2):
        for l in range(5):
            for k in range(4):
                assert torch.equal(out2[k][l][i:i + 1], single[i][k][l]), (i, l, k)
        assert torch.equal(out2[4][i:i + 1], single[i][4])
    assert not torch.equal(single[0][0][0], single[1][0][0])          # earlier outputs were not overwritten by later passes
    other = tuple(torch.randn(1, 256, h + 1, w + 2, generator=g).cuda() for h, w in sizes)
    head(other)
    assert head._engine(f2) is eng_a and head._wcache is wcache and len(head._engines) == 2
    with torch.no_grad():
        head.fcos_cls.bias.add_(1.0)                                   # parameter change -> caches are rebuilt
    assert head._engine(f2) is not eng_a


def test_registry_hooks_replace_reference_entries():
    """registry.register(force=True) / register_ops() against the UNMODIFIED reference package (imported through
    tests/golden/_ref_import.py, build container only): `type='SipMaskHead'` then builds the drop-in class, the reference
    detector's bbox_head is ours, and mmdet.ops.{CropSplit, DeformConv, nms} point at the sm_100a operators."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden'))
    import _ref_import
    if not os.path.isdir(_ref_import.REF_MM):
        pytest.skip('needs the unmodified reference mmdet package (%s), which is not present here' % _ref_import.REF_MM)
    _ref_import.install()
    from mmdet.models import build_detector
    from mmdet.models.registry import HEADS
    from sipmask_b200 import head as H
    from sipmask_b200 import ops, registry
    ref_cls, ref_fcos = HEADS.module_dict['SipMaskHead'], HEADS.module_dict['FCOSHead']
    assert ref_cls is not H.SipMaskHead
    with pytest.raises(KeyError):
        registry.register(force=False)                                  # duplicate names raise (utils/registry.py:39-42)
    registry.register(force=True)
    try:
        assert HEADS.module_dict['SipMaskHead'] is H.SipMaskHead and HEADS.module_dict['FCOSHead'] is H.FCOSHead
        model = dict(
            type='SipMask', pretrained=None,
            backbone=dict(type='ResNet', depth=50, num_stages=4, out_indices=(0, 1, 2, 3), frozen_stages=1,
                          norm_cfg=dict(type='BN', requires_grad=False), style='caffe'),
            neck=dict(type='FPN', in_channels=[256, 512, 1024, 2048], out_channels=256, start_level=1, add_extra_convs=True,
                      extra_convs_on_inputs=False, num_outs=5, relu_before_extra_convs=True),
            bbox_head=dict(type='SipMaskHead', num_classes=81, in_channels=256, stacked_convs=4, feat_channels=256,
                           strides=[8, 16, 32, 64, 128],
                           loss_cls=dict(type='FocalLoss', use_sigmoid=True, gamma=2.0, alpha=0.25, loss_weight=1.0),
                           loss_bbox=dict(type='IoULoss', loss_weight=1.0),
                           loss_centerness=dict(type='CrossEntropyLoss', use_sigmoid=True, loss_weight=1.0)))
        det = build_detector(model, train_cfg=None, test_cfg=None)
        assert type(det.bbox_head) is H.SipMaskHead
        r = det.load_state_dict(synth.detector_state_dict(50, seed=1), strict=True)      # reference-keyed checkpoint loads unchanged
        assert not r.missing_keys and not r.unexpected_keys
        import mmdet.ops as mmops
        registry.register_ops()
        assert mmops.CropSplit is ops.CropSplit and mmops.DeformConv is ops.DeformConv and mmops.nms is ops.nms
    finally:
        HEADS._module_dict['SipMaskHead'] = ref_cls
        HEADS._module_dict['FCOSHead'] = ref_fcos


@pytest.mark.gpu
def test_fcos_head_forward_matches_torch():
    import torch.nn.functional as F
    from sipmask_b200.head import FCOSHead
    torch.manual_seed(0)
    head = FCOSHead(num_classes=81, in_channels=256, stacked_convs=4, strides=[8, 16, 32, 64, 128])
    for p in head.parameters():
        if p.dim() == 4:
            torch.nn.init.normal_(p, 0, (2.0 / (p.shape[1] * p.shape[2] * p.shape[3])) ** 0.5)
    head = head.cuda()
    feats = tuple(torch.randn(1, 256, h, w, device='cuda') for h, w in [(12, 16), (6, 8), (3, 4), (2, 2), (1, 1)])
    cls, box, ctr = head(feats)
    for l, x in enumerate(feats):
        c = r = x
        for m in head.cls_convs:
            c = F.relu(F.group_norm(F.conv2d(c, m.conv.weight, None, padding=1), 32, m.gn.weight, m.gn.bias))
        for m in head.reg_convs:
            r = F.relu(F.group_norm(F.conv2d(r, m.conv.weight, None, padding=1), 32, m.gn.weight, m.gn.bias))
        ref_cls = F.conv2d(c, head.fcos_cls.weight, head.fcos_cls.bias, padding=1)
        ref_ctr = F.conv2d(c, head.fcos_centerness.weight, head.fcos_centerness.bias, padding=1)
        ref_box = (F.conv2d(r, head.fcos_reg.weight, head.fcos_reg.bias, padding=1) * head.scales[l].scale).exp()
        for a, b in ((cls[l], ref_cls), (ctr[l], ref_ctr), (box[l], ref_box)):
            assert a.shape == b.shape
            assert ((a - b).norm() / (b.norm() + 1e-9)).item() < 3e-2
