"""GPU parity tests for the tcgen05 implicit-GEMM convolution and the NHWC helper kernels (run with -m gpu).
References are plain PyTorch ops in float64 on the fp16-rounded operands (the fp32-accumulating tensor-core result
must then agree to fp16 output rounding)."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _nhwc(x):      # NCHW -> NHWC fp16 contiguous (cuda)
    return x.permute(0, 2, 3, 1).contiguous().to(torch.float16).cuda()


def _ref_conv(x16, w16, k, stride, bias=None, residual=None, relu=False, alpha=1.0):
    """x16 NHWC fp16 (cuda), w16 packed [Cout, k*k*Cin] fp16 -> NHWC float64 reference."""
    N, H, W, C = x16.shape
    cout = w16.shape[0]
    w = w16.double().view(cout, k, k, C).permute(0, 3, 1, 2)
    y = F.conv2d(x16.double().permute(0, 3, 1, 2), w, stride=stride, padding=k // 2)
    if bias is not None:
        y = y + bias.double().view(1, -1, 1, 1)
    y = y * alpha
    y = y.permute(0, 2, 3, 1)
    if residual is not None:
        y = y + residual.double()
    if relu:
        y = y.clamp(min=0)
    return y


def _check(out, ref, tol=2e-3):
    out = out.double()
    err = (out - ref).abs().max().item()
    scale = ref.abs().max().item() + 1e-6
    assert err <= tol * scale + 1e-3, 'max abs err %g (scale %g)' % (err, scale)


@pytest.mark.parametrize('H,W,cin,cout,k,stride', [
    (8, 160, 128, 256, 1, 1),       # plain GEMM: M=1280, K=128, N=256
    (25, 42, 64, 64, 1, 1),         # N tile 64, ragged M tiles
    (13, 21, 256, 2048, 1, 1),      # 8 N tiles
    (25, 42, 256, 256, 3, 1),       # 3x3, TMA zero-fill padding, 36 k-blocks
    (7, 11, 256, 256, 3, 1),        # one ragged tile
    (100, 168, 256, 256, 3, 1),     # P3 tower conv (full size)
    (25, 42, 256, 256, 3, 2),       # FPN P6: stride 2, odd H -> parity maps
    (13, 21, 256, 256, 3, 2),       # FPN P7: odd H and W
    (50, 84, 256, 512, 1, 2),       # caffe-style strided 1x1
    (25, 42, 512, 128, 1, 1),
    (20, 20, 768, 512, 1, 1),       # sip_mask_lat0
    (9, 5, 2304, 256, 1, 1),        # DCN GEMM (K = 9*256)
    (104, 208, 256, 256, 3, 1),     # 169 M-tiles (odd): 2-CTA clusters multicast the weight tile, last cluster has a dummy CTA
    (200, 336, 64, 256, 1, 1),      # layer1 conv3 shape: 525 M-tiles, one k-block, cluster path
    (120, 160, 128, 512, 3, 1),     # 2 N-tiles x 150 M-tiles
])
def test_conv_matches_reference(H, W, cin, cout, k, stride):
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(H * 1000 + W + cin + cout)
    x = _nhwc(torch.randn(2 if H < 50 else 1, cin, H, W, generator=g))
    w = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
    wk, _ = conv.pack_weight(w, device='cuda')
    Ho, Wo = (H + 2 * (k // 2) - k) // stride + 1, (W + 2 * (k // 2) - k) // stride + 1
    out = torch.full((x.shape[0], Ho, Wo, cout), float('nan'), dtype=torch.float16, device='cuda')
    plan = conv.ConvPlan(x, wk, out, k, stride)
    plan.run()
    torch.cuda.synchronize()
    assert torch.isfinite(out.float()).all()
    _check(out, _ref_conv(x, wk, k, stride))
    # running twice must give the same answer (barrier phases / TMEM reuse)
    out2 = out.clone()
    plan.run()
    torch.cuda.synchronize()
    assert torch.equal(out, out2)


def test_conv_epilogue_bias_residual_relu_gnstats():
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(5)
    N, H, W, C = 2, 25, 42, 256
    x = _nhwc(torch.randn(N, C, H, W, generator=g))
    w = torch.randn(C, C, 3, 3, generator=g) / 48.0
    bn = (torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1, torch.randn(C, generator=g) * 0.1,
          torch.rand(C, generator=g) + 0.5)
    wk, bias = conv.pack_weight(w, bn=bn, device='cuda')
    res = _nhwc(torch.randn(N, C, H, W, generator=g))
    out = torch.empty((N, H, W, C), dtype=torch.float16, device='cuda')
    stats = torch.zeros((N, 32, 2), dtype=torch.int64, device='cuda')
    plan = conv.ConvPlan(x, wk, out, 3, 1, relu=True, bias=bias, residual=res, gn_stats=stats)
    plan.run()
    torch.cuda.synchronize()
    pre = _ref_conv(x, wk, 3, 1, bias=bias, residual=res, relu=False)
    _check(out, pre.clamp(min=0))
    # GN statistics are taken on the pre-activation value (conv + bias + residual), per (image, 8-channel group)
    grp = pre.view(N, H * W, 32, 8)
    np.testing.assert_allclose(stats[:, :, 0].double().cpu().numpy() / 2 ** 20, grp.sum((1, 3)).cpu().numpy(), rtol=2e-3, atol=0.5)
    np.testing.assert_allclose(stats[:, :, 1].double().cpu().numpy() / 2 ** 16, (grp * grp).sum((1, 3)).cpu().numpy(), rtol=2e-3, atol=0.5)
    s1 = stats.clone()
    stats.zero_()
    plan.run()
    torch.cuda.synchronize()
    assert torch.equal(stats, s1)          # integer atomics: bit-reproducible
    # folded BN == eval BatchNorm of the reference (resnet.py:514-521)
    y = F.conv2d(x.float().permute(0, 3, 1, 2), w.cuda(), padding=1)
    y = F.batch_norm(y, bn[2].cuda(), bn[3].cuda(), bn[0].cuda(), bn[1].cuda(), False, 0.0, 1e-5)
    y = (y.permute(0, 2, 3, 1) + res.float()).clamp(min=0)
    _check(out, y.double(), tol=5e-3)


def test_conv_fp32_heads_alpha_and_fpn_residual():
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(6)
    x = _nhwc(torch.randn(1, 256, 13, 21, generator=g))
    for cout, alpha in ((16, 1.3), (208, 1.0)):
        w = torch.randn(cout, 256, 3, 3, generator=g) / 48.0
        b = torch.randn(cout, generator=g).cuda()
        wk, _ = conv.pack_weight(w, device='cuda')
        out = torch.empty((1, 13, 21, cout), dtype=torch.float32, device='cuda')
        conv.ConvPlan(x, wk, out, 3, 1, bias=b, alpha=alpha).run()
        torch.cuda.synchronize()
        _check(out, _ref_conv(x, wk, 3, 1, bias=b, alpha=alpha), tol=1e-4)
    # FPN lateral: 1x1 conv + bias + nearest-upsampled coarser level (fpn.py:149-152), incl. non-x2 sizes
    for (H, W, rh, rw) in ((26, 42, 13, 21), (25, 41, 13, 21)):
        xin = _nhwc(torch.randn(1, 512, H, W, generator=g))
        coarse = _nhwc(torch.randn(1, 256, rh, rw, generator=g))
        w = torch.randn(256, 512, 1, 1, generator=g) / 22.0
        b = torch.randn(256, generator=g).cuda()
        wk, _ = conv.pack_weight(w, device='cuda')
        out = torch.empty((1, H, W, 256), dtype=torch.float16, device='cuda')
        conv.ConvPlan(xin, wk, out, 1, 1, bias=b, residual=coarse, residual_upsample=True).run()
        torch.cuda.synchronize()
        up = F.interpolate(coarse.float().permute(0, 3, 1, 2), size=(H, W), mode='nearest').permute(0, 2, 3, 1)
        _check(out, _ref_conv(xin, wk, 1, 1, bias=b, residual=up))


@pytest.mark.parametrize('H,W', [(64, 96), (160, 224)])
def test_stem_matches_reference(H, W):
    from sipmask_b200 import conv, synth
    g = torch.Generator().manual_seed(7)
    img = synth.synthetic_image(H, W, batch=2, seed=1).cuda()
    w = torch.randn(64, 3, 7, 7, generator=g) * 0.01
    bn = (torch.rand(64, generator=g) + 0.5, torch.randn(64, generator=g) * 0.1, torch.randn(64, generator=g) * 0.1,
          torch.rand(64, generator=g) + 0.5)
    wk, bias = conv.pack_stem_weight(w, bn, device='cuda')
    img8 = conv.image_to_nhwc8(img)
    out = torch.empty((2, H // 2, W // 2, 64), dtype=torch.float16, device='cuda')
    conv.StemPlan(img8, wk, bias, out, 2, H, W).run()
    torch.cuda.synchronize()
    s = (bn[0] / torch.sqrt(bn[3] + 1e-5)).cuda()
    wq = (w.cuda() * s.view(-1, 1, 1, 1)).half().double()
    y = F.conv2d(img.half().double(), wq, stride=2, padding=3) + bias.double().view(1, -1, 1, 1)
    _check(out, y.clamp(min=0).permute(0, 2, 3, 1))
    # space-to-depth form (K = 256): same convolution, same fp16 weights, different summation grouping only
    wk2, bias2 = conv.pack_stem_weight_s2d(w, bn, device='cuda')
    q = conv.image_to_s2d16(img)
    assert q.shape == (2, H // 2 + 3, W // 2 + 4, 16)
    p8 = img8.float()                                           # [2, H+6, W+8, 8]: padded pixels, channels 0..2 real
    want_q = p8.view(2, H // 2 + 3, 2, W // 2 + 4, 2, 8)[..., :4].permute(0, 1, 3, 2, 4, 5).reshape(2, H // 2 + 3, W // 2 + 4, 16)
    assert torch.equal(q.float(), want_q)                       # q(Y, X, (dy*2+dx)*4 + c) = padded pixel (2Y+dy, 2X+dx, c)
    out2 = torch.empty_like(out)
    conv.StemPlan(q, wk2, bias2, out2, 2, H, W, s2d=True).run()
    torch.cuda.synchronize()
    _check(out2, y.clamp(min=0).permute(0, 2, 3, 1))
    # max pool 3x3/2 pad 1 (resnet.py:460)
    mp = conv.maxpool3x3s2(out)
    ref = F.max_pool2d(out.float().permute(0, 3, 1, 2), 3, 2, 1).permute(0, 2, 3, 1)
    assert torch.equal(mp.float(), ref)


def test_groupnorm_kernels():
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(8)
    x = _nhwc(torch.randn(2, 256, 13, 21, generator=g) * 2 + 0.5)
    gamma = (torch.rand(256, generator=g) + 0.5).cuda()
    beta = torch.randn(256, generator=g).cuda()
    stats = conv.groupnorm_stats(x)
    ref = F.relu(F.group_norm(x.float().permute(0, 3, 1, 2), 32, gamma, beta, 1e-5)).permute(0, 2, 3, 1)
    y = conv.groupnorm_relu_apply(x.clone(), stats, gamma, beta)
    torch.cuda.synchronize()
    _check(y, ref.double(), tol=3e-3)


def test_deform_im2col_and_offsets_match_oracle():
    from oracle import ops as O
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(9)
    N, C, H, W = 2, 256, 13, 21
    x = torch.randn(N, C, H, W, generator=g)
    bbox = torch.randn(N, 4, H, W, generator=g) * 3
    w_off = torch.randn(72, 4, 1, 1, generator=g) * 0.3
    scale = 1.2
    off_ref = F.conv2d(bbox * scale, w_off)                                     # FeatureAlign.conv_offset
    x16 = x.half()
    cols_ref, _, _ = O.deform_im2col(x16.float(), off_ref, 3, 3, 1, 1, 1, 4)    # [N, C*9, HW], row = c*9 + tap
    cols_ref = cols_ref.view(N, C, 9, H * W).permute(0, 3, 2, 1).reshape(N, H, W, 9 * C)   # -> [.., tap*C + c]
    bb = bbox.permute(0, 2, 3, 1).contiguous().cuda()
    off = conv.offset_conv1x1(bb, scale, w_off.view(72, 4).contiguous().cuda())
    np.testing.assert_allclose(off.cpu().numpy(), off_ref.permute(0, 2, 3, 1).numpy(), rtol=1e-5, atol=1e-5)
    col = conv.deform_im2col(_nhwc(x), off, 4)
    torch.cuda.synchronize()
    _check(col, cols_ref.double().cuda(), tol=2e-3)


def test_upsample_bilinear_matches_torch():
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(10)
    x = _nhwc(torch.randn(1, 256, 13, 21, generator=g))
    for f in (2, 4):
        ref = F.interpolate(x.float().permute(0, 3, 1, 2), scale_factor=f, mode='bilinear', align_corners=False)
        out = torch.zeros((1, 13 * f, 21 * f, 768), dtype=torch.float16, device='cuda')
        conv.upsample_bilinear(x, f, out=out, out_choff=256)
        torch.cuda.synchronize()
        _check(out[..., 256:512], ref.permute(0, 2, 3, 1).double(), tol=2e-3)
        assert out[..., :256].abs().max() == 0 and out[..., 512:].abs().max() == 0
        # an output smaller than the upsampled map (a P3 map that is not exactly 2x / 4x the level): the top-left crop,
        # and nothing written past the output
        ho, wo = 13 * f - f + 1, 21 * f - 3
        buf = torch.zeros(ho * wo * 768 + 4096, dtype=torch.float16, device='cuda')
        out = buf[:ho * wo * 768].view(1, ho, wo, 768)
        conv.upsample_bilinear(x, f, out=out, out_choff=256)
        torch.cuda.synchronize()
        _check(out[..., 256:512], ref[:, :, :ho, :wo].permute(0, 2, 3, 1).double(), tol=2e-3)
        assert buf[ho * wo * 768:].abs().max() == 0
    out = torch.zeros((1, 13, 21, 768), dtype=torch.float16, device='cuda')
    conv.upsample_bilinear(x, 1, out=out, out_choff=0)
    assert torch.equal(out[..., :256], x)


def test_multi_level_conv_and_helpers_match_single_level():
    """One launch over five pyramid levels == five single-level launches, bit for bit (shared tower weights)."""
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(11)
    sizes = [(25, 42), (13, 21), (7, 11), (4, 6), (2, 3)]
    xs = [_nhwc(torch.randn(1, 256, h, w, generator=g)) for h, w in sizes]
    w = torch.randn(256, 256, 3, 3, generator=g) / 48.0
    wk, _ = conv.pack_weight(w, device='cuda')
    st_m = [torch.zeros((1, 32, 2), dtype=torch.int64, device='cuda') for _ in sizes]
    outs = [torch.empty((1, h, w_, 256), dtype=torch.float16, device='cuda') for h, w_ in sizes]
    conv.ConvPlanMulti(xs, wk, outs, 3, gn_stats=st_m).run()
    gamma = (torch.rand(256, generator=g) + 0.5).cuda()
    beta = torch.randn(256, generator=g).cuda()
    raw = [o.clone() for o in outs]
    conv.groupnorm_relu_apply_multi(outs, st_m, gamma, beta)
    torch.cuda.synchronize()
    for i, (h, w_) in enumerate(sizes):
        st = torch.zeros((1, 32, 2), dtype=torch.int64, device='cuda')
        o = torch.empty((1, h, w_, 256), dtype=torch.float16, device='cuda')
        conv.ConvPlan(xs[i], wk, o, 3, 1, gn_stats=st).run()
        torch.cuda.synchronize()
        assert torch.equal(o, raw[i]) and torch.equal(st, st_m[i]), i
        _check(o, _ref_conv(xs[i], wk, 3, 1))
        conv.groupnorm_relu_apply(o, st, gamma, beta)
        torch.cuda.synchronize()
        assert (o.float() - outs[i].float()).abs().max().item() <= 2e-3 * (o.float().abs().max().item() + 1)
    # fp32 multi-level heads with bias into pitch-208 / pitch-16 slices of level-concatenated buffers
    tot = sum(h * w_ for h, w_ in sizes)
    big = torch.zeros((1, tot, 208), dtype=torch.float32, device='cuda')
    offs0 = [sum(h * w_ for h, w_ in sizes[:l]) for l in range(len(sizes))]
    views = [big[:, offs0[l]:offs0[l] + sizes[l][0] * sizes[l][1]].view(1, sizes[l][0], sizes[l][1], 208) for l in range(len(sizes))]
    w2 = torch.randn(208, 256, 3, 3, generator=g) / 48.0
    b2 = torch.randn(208, generator=g).cuda()
    wk2, _ = conv.pack_weight(w2, device='cuda')
    conv.ConvPlanMulti(xs, wk2, views, 3, bias=b2).run()
    torch.cuda.synchronize()
    for i in range(len(sizes)):
        _check(views[i], _ref_conv(xs[i], wk2, 3, 1, bias=b2), tol=1e-4)
    # batched offsets + deformable im2col == per-level kernels
    bbs = [torch.randn(1, h, w_, 16, generator=g).cuda() * 3 for h, w_ in sizes]
    scales = [1.0, 1.1, 1.2, 1.3, 1.4]
    w_off = (torch.randn(72, 4, generator=g) * 0.3).cuda()
    offs = [torch.empty((1, h, w_, 72), dtype=torch.float32, device='cuda') for h, w_ in sizes]
    cols = [torch.empty((1, h, w_, 2304), dtype=torch.float16, device='cuda') for h, w_ in sizes]
    conv.offset_conv1x1_multi(bbs, scales, w_off, offs)
    conv.deform_im2col_multi(xs, offs, 4, cols)
    torch.cuda.synchronize()
    for i in range(len(sizes)):
        o1 = conv.offset_conv1x1(bbs[i], scales[i], w_off)
        c1 = conv.deform_im2col(xs[i], o1, 4)
        torch.cuda.synchronize()
        assert torch.equal(o1, offs[i]), i
        # the batched kernel evaluates the four bilinear terms in one expression (different FMA contraction): fp16-ulp level
        assert (c1.float() - cols[i].float()).abs().max().item() <= 2e-3 * (c1.float().abs().max().item() + 1), i


@pytest.mark.parametrize('H,W,cin,cout,stride,res', [(200, 336, 64, 256, 1, True), (50, 84, 256, 512, 2, False),
                                                     (13, 21, 256, 2048, 1, True), (8, 160, 128, 256, 1, False)])
def test_small_1x1_kernel_matches_persistent_kernel(H, W, cin, cout, stride, res, monkeypatch):
    """conv1x1_small_kernel (one 128 x 128 tile per CTA, 2-3 CTAs per SM; SMB_CONV_SMALL=1) is an alternative execution of the
    short-K 1x1 convolutions: bit-identical to the persistent kernel (same MMA order over K, same epilogue arithmetic)."""
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(H + cout)
    x = _nhwc(torch.randn(1, cin, H, W, generator=g))
    w = torch.randn(cout, cin, 1, 1, generator=g) / (cin ** 0.5)
    wk, _ = conv.pack_weight(w, device='cuda')
    bias = torch.randn(cout, generator=g).cuda()
    Ho, Wo = (H - 1) // stride + 1, (W - 1) // stride + 1
    r = _nhwc(torch.randn(1, cout, Ho, Wo, generator=g)) if res else None
    outs = []
    for small in ('0', '1'):
        monkeypatch.setenv('SMB_CONV_SMALL', small)
        out = torch.zeros((1, Ho, Wo, cout), dtype=torch.float16, device='cuda')
        conv.ConvPlan(x, wk, out, 1, stride, relu=True, bias=bias, residual=r).run()
        torch.cuda.synchronize()
        outs.append(out)
    assert torch.equal(outs[0], outs[1])
    _check(outs[1], _ref_conv(x, wk, 1, stride, bias=bias, residual=r, relu=True))


@pytest.mark.parametrize('H,W,cin,cout,k,stride,res', [(200, 336, 64, 256, 1, 1, True), (100, 168, 256, 64, 1, 1, False),
                                                       (50, 84, 256, 512, 1, 2, False), (25, 42, 256, 256, 3, 1, False),
                                                       (13, 21, 512, 2048, 1, 1, True), (37, 53, 128, 128, 3, 1, False)])
def test_split_epilogue_matches_lockstep_epilogue(H, W, cin, cout, k, stride, res, monkeypatch):
    """epilogue_split (the two warp groups drain alternate 64-channel chunks) against the lockstep epilogue of the same kernel
    (SMB_CONV_EPI_SPLIT=0): the per-element arithmetic (acc + bias, + residual, ReLU, round) is the same sequence, so the
    outputs are bit-identical."""
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(H * 3 + cout + k)
    x = _nhwc(torch.randn(1, cin, H, W, generator=g))
    w = torch.randn(cout, cin, k, k, generator=g) / ((cin * k * k) ** 0.5)
    wk, _ = conv.pack_weight(w, device='cuda')
    bias = torch.randn(cout, generator=g).cuda()
    Ho, Wo = (H + 2 * (k // 2) - k) // stride + 1, (W + 2 * (k // 2) - k) // stride + 1
    r = _nhwc(torch.randn(1, cout, Ho, Wo, generator=g)) if res else None
    outs = []
    for split in ('0', '1'):
        monkeypatch.setenv('SMB_CONV_EPI_SPLIT', split)
        out = torch.zeros((1, Ho, Wo, cout), dtype=torch.float16, device='cuda')
        conv.ConvPlan(x, wk, out, k, stride, relu=True, bias=bias, residual=r).run()
        torch.cuda.synchronize()
        outs.append(out)
    for o in outs[1:]:
        assert torch.equal(outs[0], o)
    _check(outs[0], _ref_conv(x, wk, k, stride, bias=bias, residual=r, relu=True))
