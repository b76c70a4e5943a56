"""Every convolution plan the engine builds, checked per element against a float64 reference (run with -m gpu).

Each case is named for the planner branch it targets (conv_tcgen05.cu finish_plan: N tile, cta_group::2 pair mode, TMA-store
or direct epilogue, TMA-staged residual, split or lockstep epilogue) and asserts that branch through ConvPlan.info(), so a
change of the planner's heuristics cannot silently drop coverage: if a case stops landing on its branch, change its shape.

Reference: F.conv2d in float64 on the fp16 operands, then bias, x alpha, + residual, ReLU.  Per-element bound: with
A = |x| (*) |w| (a second float64 convolution of the absolute values) and K the reduction length,
    B = |alpha| * 2^-22 * (K * A + |bias|)
i.e. twice the round-to-nearest bound of a K-term fp32 accumulation (the tensor core's adder may truncate) plus the fp32
roundings of the epilogue.  fp16 outputs must satisfy |out - ref| <= ulp16(|ref| + B) + B, fp32 outputs
|out - ref| <= 2^-23 |ref| + B.  Every output is a view into a larger buffer filled with a sentinel, and every GroupNorm
statistics buffer has one extra image: whatever lies outside the views must be untouched afterwards.

Schedule invariance: the outputs and statistics of every case are bit-identical across plan variants (grid caps, widest /
narrowest N tile, pair mode off, a second run): each output element accumulates K in the same order whatever the tiling, and
the statistics are integer sums of the same fixed-point partials."""
import zlib

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

SENTINEL = 0x7E01            # an fp16 NaN payload the kernels never produce; compared as int16
GAMMA_256 = 256 * 2.0 ** -24 / (1 - 256 * 2.0 ** -24)     # fp32 summation bound of the in-warp statistics partials
GN_SUM_Q, GN_SQ_Q = 2.0 ** -21, 2.0 ** -17                # half a fixed-point quantum per statistics atomic (2^20, 2^16)


def _tiles(H, W):
    """M tiles of one image of an H x W output (conv_tcgen05.cu choose_patch: the BH x BW = 128 patch with fewest tiles)."""
    return min(-(-H // bh) * -(-W // bw) for bh, bw in ((1, 128), (2, 64), (4, 32), (8, 16), (16, 8)))


def _ulp16(v):
    return torch.exp2(torch.floor(torch.log2(v.clamp(min=2.0 ** -14))) - 10)


class Guarded(object):
    """One allocation filled with the sentinel; views into it are kernel outputs, everything else must survive a run."""

    def __init__(self, numel, dtype):
        self.per = torch.empty(0, dtype=dtype).element_size() // 2
        self.buf16 = torch.full((numel * self.per,), SENTINEL, dtype=torch.int16, device='cuda')
        self.data = self.buf16.view(dtype)
        self.mark = torch.zeros(numel, dtype=torch.bool, device='cuda')

    def view(self, offset, N, H, W, pitch, choff, C):
        n = N * H * W * pitch
        self.mark[offset:offset + n].view(N, H, W, pitch)[..., choff:choff + C] = True
        return self.data[offset:offset + n].view(N, H, W, pitch)[..., choff:choff + C]

    def reset(self):
        self.buf16.fill_(SENTINEL)

    def clobbered(self):
        return int((self.buf16.view(-1, self.per)[~self.mark] != SENTINEL).sum())


def _bits(t):
    return t.contiguous().view(torch.int16 if t.dtype == torch.float16 else torch.int32)


class Case(object):
    """Inputs, guarded outputs, statistics buffers and the float64 reference of one convolution plan."""

    def __init__(self, name, N, sizes, cin, cout, k, stride=1, bias=False, residual=None, res_hw=None, relu=False, alpha=1.0,
                 out_dtype=torch.float16, gn=False, in_pitch=None, in_off=0, out_pitch=None, out_off=0, bias_offset=0,
                 cout_real=None, multi=False, gap=37, expect=None):
        self.name, self.N, self.k, self.stride, self.relu, self.alpha, self.multi = name, N, k, stride, relu, alpha, multi
        self.expect = expect or {}
        g = torch.Generator().manual_seed(zlib.crc32(name.encode()))
        in_pitch = in_pitch or cin
        self.xs = []
        for (H, W) in sizes:
            xb = torch.randn(N, H, W, in_pitch, generator=g).half().cuda()
            self.xs.append(xb[..., in_off:in_off + cin])
        w = torch.randn(cout, cin, k, k, generator=g) / (cin * k * k) ** 0.5
        if cout_real is not None:
            w[cout_real:] = 0
        from sipmask_b200 import conv
        self.wk, _ = conv.pack_weight(w, device='cuda')
        self.bias = None
        if bias:
            b = torch.randn(cout, generator=g)
            if cout_real is not None:
                b[cout_real:] = 0
            store = torch.zeros(cout + 4, device='cuda')
            self.bias = store[bias_offset:bias_offset + cout]          # bias_offset = 1: 4 bytes off 16-byte alignment
            self.bias.copy_(b)
        outs = [((H + 2 * (k // 2) - k) // stride + 1, (W + 2 * (k // 2) - k) // stride + 1) for H, W in sizes]
        self.out_sizes = outs
        self.residual = None
        if residual == 'same':
            self.residual = torch.randn(N, outs[0][0], outs[0][1], cout, generator=g).half().cuda()
        elif residual == 'up':
            self.residual = torch.randn(N, res_hw[0], res_hw[1], cout, generator=g).half().cuda()
        # outputs: level-major views into one sentinel-filled buffer, a gap of `gap` pixels before, between and after them
        out_pitch = out_pitch or cout
        offs, o = [], gap * out_pitch
        for (h, w_) in outs:
            offs.append(o)
            o += (N * h * w_ + gap) * out_pitch
        self.guard = Guarded(o, out_dtype)
        self.outs = [self.guard.view(off, N, h, w_, out_pitch, out_off, cout) for off, (h, w_) in zip(offs, outs)]
        self.stats_full = [torch.zeros((N + 1, 32, 2), dtype=torch.int64, device='cuda') for _ in outs] if gn else None
        self.stats = [s[:N] for s in self.stats_full] if gn else None
        self._reference()

    def _reference(self):
        N, k, cout = self.N, self.k, self.wk.shape[0]
        cin = self.xs[0].shape[3]
        wd = self.wk.double().view(cout, k, k, cin).permute(0, 3, 1, 2)
        K = k * k * cin
        self.pre, self.post, self.B = [], [], []
        for x in self.xs:
            xd = x.double().permute(0, 3, 1, 2)
            c = F.conv2d(xd, wd, stride=self.stride, padding=k // 2).permute(0, 2, 3, 1)
            a = F.conv2d(xd.abs(), wd.abs(), stride=self.stride, padding=k // 2).permute(0, 2, 3, 1)
            babs = 0.0
            if self.bias is not None:
                c = c + self.bias.double()
                babs = self.bias.double().abs()
            c = c * self.alpha
            B = abs(self.alpha) * 2.0 ** -22 * (K * a + babs)
            if self.residual is not None:
                r = self.residual.double()
                if r.shape[1:3] != c.shape[1:3]:          # F.interpolate(mode='nearest', size=...) as fpn.py:149-152
                    r = F.interpolate(r.permute(0, 3, 1, 2), size=c.shape[1:3], mode='nearest').permute(0, 2, 3, 1)
                c = c + r
            self.pre.append(c)
            self.post.append(c.clamp(min=0) if self.relu else c)
            self.B.append(B)

    def new_plan(self):
        from sipmask_b200 import conv
        if self.multi:
            return conv.ConvPlanMulti(self.xs, self.wk, self.outs, self.k, relu=self.relu, bias=self.bias, gn_stats=self.stats,
                                      alpha=self.alpha)
        return conv.ConvPlan(self.xs[0], self.wk, self.outs[0], self.k, self.stride, relu=self.relu, bias=self.bias,
                             residual=self.residual, residual_upsample=self.residual is not None and
                             self.residual.shape[1:3] != self.outs[0].shape[1:3],
                             gn_stats=self.stats[0] if self.stats else None, alpha=self.alpha)

    def run(self, plan):
        self.guard.reset()
        if self.stats_full:
            for s in self.stats_full:
                s.zero_()
        plan.run()
        torch.cuda.synchronize()

    def guard_problems(self, what):
        bad = []
        if self.guard.clobbered():
            bad.append('%s: %d sentinel elements outside the output views overwritten' % (what, self.guard.clobbered()))
        for l, s in enumerate(self.stats_full or []):
            tail = s[self.N:].view(-1)
            if int((tail != 0).sum()):
                bad.append('%s: level %d wrote %d statistics slots past image %d, e.g. %s' % (
                    what, l, int((tail != 0).sum()), self.N - 1, tail[:6].tolist()))
        return bad

    def check_guards(self, what):
        bad = self.guard_problems(what)
        assert not bad, '\n'.join(bad)

    def snapshot(self):
        return [_bits(o) for o in self.outs] + ([s.clone() for s in self.stats_full] if self.stats_full else [])


def _out_bound(out, ref, B):
    if out.dtype == torch.float16:
        return _ulp16(ref.abs() + B) + B
    return 2.0 ** -23 * ref.abs() + B


def _check_elements(case):
    worst = 0.0
    for l, (o, ref, B) in enumerate(zip(case.outs, case.post, case.B)):
        assert torch.isfinite(o).all(), '%s level %d: non-finite output' % (case.name, l)
        err = (o.double() - ref).abs()
        bound = _out_bound(o, ref, B)
        bad = int((err > bound).sum())
        ratio = (err / bound.clamp(min=1e-300)).max().item()
        worst = max(worst, ratio)
        assert bad == 0, '%s level %d: %d elements out of bound, worst err/bound %.3g' % (case.name, l, bad, ratio)
    return worst


def _stats_bounds(case, l):
    """fp64 reference sums and error bounds of the per-(image, group) statistics of level l."""
    pre, B = case.pre[l], case.B[l]
    N, H, W, C = pre.shape
    cpg = C // 32
    grp = lambda t: t.reshape(N, H * W, 32, cpg)
    S_ref, Q_ref = grp(pre).sum((1, 3)), grp(pre * pre).sum((1, 3))
    mag = grp(pre.abs() + B)
    n_atomics = _tiles(H, W) * 4 * (cpg // 8)        # one atomic per (M tile, 32-row lane quadrant, 8-channel partial)
    S_err = grp(B).sum((1, 3)) + GAMMA_256 * mag.sum((1, 3)) + n_atomics * GN_SUM_Q
    Q_err = grp(B * (2 * pre.abs() + B)).sum((1, 3)) + GAMMA_256 * (mag * mag).sum((1, 3)) + n_atomics * GN_SQ_Q
    return S_ref, Q_ref, S_err, Q_err


def _check_stats(case):
    """Worst err/bound of the per-(image, group) sums and sums of squares, and a message per failing (level, kind)."""
    worst, bad = 0.0, []
    for l, st in enumerate(case.stats):
        S_ref, Q_ref, S_err, Q_err = _stats_bounds(case, l)
        S = st[..., 0].double() / 2 ** 20
        Q = st[..., 1].double() / 2 ** 16
        for what, got, ref, bound in (('sum', S, S_ref, S_err), ('sumsq', Q, Q_ref, Q_err)):
            err = (got - ref).abs()
            ratio = (err / bound).max().item()
            worst = max(worst, ratio)
            if not (err <= bound).all():
                bad.append('%s level %d GN %s: %d of %d (image, group) values out of bound, worst err/bound %.3g; got %s want %s'
                           % (case.name, l, what, int((err > bound).sum()), err.numel(), ratio,
                              ['%.6g' % v for v in got[err > bound][:4].tolist()],
                              ['%.6g' % v for v in ref[err > bound][:4].tolist()]))
    return worst, bad


def _check_gn_apply(case):
    """groupnorm_relu_apply_multi on the kernel's statistics vs fp64 GroupNorm(32) + ReLU of the reference pre-activation."""
    from sipmask_b200 import conv
    g = torch.Generator().manual_seed(zlib.crc32(case.name.encode()) + 1)
    C = case.wk.shape[0]
    gamma = (torch.rand(C, generator=g) + 0.5).cuda()
    beta = torch.randn(C, generator=g).cuda()
    ys = [o.contiguous() for o in case.outs]
    conv.groupnorm_relu_apply_multi(ys, case.stats, gamma, beta, 1e-5, True)
    torch.cuda.synchronize()
    worst = 0.0
    for l, (y, pre, B) in enumerate(zip(ys, case.pre, case.B)):
        N, H, W, _ = pre.shape
        cpg, cnt = C // 32, H * W * (C // 32)
        S_ref, Q_ref, S_err, Q_err = _stats_bounds(case, l)
        mean, ex2 = S_ref / cnt, Q_ref / cnt
        var = ex2 - mean * mean
        dmean = S_err / cnt + 2.0 ** -22 * mean.abs()           # + int64 -> fp32 conversion and the 1/count scaling
        dex2 = Q_err / cnt + 2.0 ** -22 * ex2
        dvar = dex2 + 2 * mean.abs() * dmean + dmean * dmean + 2.0 ** -23 * (ex2 + mean * mean)
        assert (var + 1e-5 - dvar > 0).all()
        rstd = (var + 1e-5).rsqrt()
        drstd = 0.5 * (var + 1e-5 - dvar) ** -1.5 * dvar + 2.0 ** -21 * rstd
        per_ch = lambda t: t.repeat_interleave(cpg, dim=1).view(N, 1, 1, C)
        mean_c, dmean_c, rstd_c, drstd_c = per_ch(mean), per_ch(dmean), per_ch(rstd), per_ch(drstd)
        ref = F.relu((pre - mean_c) * rstd_c * gamma.double() + beta.double())
        assert torch.allclose(ref, F.relu(F.group_norm(pre.permute(0, 3, 1, 2), 32, gamma.double(), beta.double(), 1e-5))
                              .permute(0, 2, 3, 1))
        e_in = _out_bound(case.outs[l], pre, B)                  # the conv output's own bound (fp16 rounding + accumulation)
        dev = (pre - mean_c).abs()
        ga = gamma.double().abs()
        d = ga * ((dev + e_in + dmean_c) * drstd_c + rstd_c * (e_in + dmean_c)) + 2.0 ** -22 * (dev * rstd_c * ga + beta.double().abs())
        bound = _ulp16(ref.abs() + d) + d
        err = (y.double() - ref).abs()
        ratio = (err / bound).max().item()
        worst = max(worst, ratio)
        assert (err <= bound).all(), '%s level %d GN apply: %d elements out of bound, worst err/bound %.3g' % (
            case.name, l, int((err > bound).sum()), ratio)
    return worst


LEVELS = [(25, 42), (13, 21), (7, 11), (4, 6), (2, 3)]
ODD_LEVELS = [(24, 40), (13, 21), (7, 11), (4, 6), (2, 3)]        # 9 + 3 + 1 + 1 + 1 = 15 M tiles per image
TMA_SPLIT = dict(pair=1, out_tma=1, epi_split=1)

CASES = {
    # bottleneck conv3 shape: short K, same-shape residual staged by TMA, the split epilogue
    'pair_tma_store_tma_residual_split_epilogue': dict(
        N=3, sizes=[(40, 56)], cin=64, cout=256, k=1, bias=True, residual='same', relu=True,
        expect=dict(TMA_SPLIT, n_tile=256, res_tma=1)),
    'strided_1x1_parity_maps_several_n_tiles': dict(
        N=3, sizes=[(27, 43)], cin=256, cout=512, k=1, stride=2, relu=True, expect=dict(pair=1, out_tma=1, n_tiles_n=8)),
    'conv3x3_bias_pair_tma_store': dict(N=3, sizes=[(25, 42)], cin=256, cout=256, k=3, bias=True, expect=TMA_SPLIT),
    'fpn_lateral_nearest_upsampled_residual': dict(
        N=3, sizes=[(25, 41)], cin=512, cout=256, k=1, bias=True, residual='up', res_hw=(13, 21),
        expect=dict(pair=1, out_tma=1, res_tma=0, epi_split=0)),
    # prototype conv sip_mask_lat (engine.py _build_head): N tile 32, direct fp16 stores
    'proto_3x3_512_to_32_pair_direct_fp16': dict(
        N=3, sizes=[(25, 42)], cin=512, cout=32, k=3, bias=True, relu=True, expect=dict(pair=1, out_tma=0, n_tile=32)),
    # DCN offset conv: 18 offsets padded to 32 channels, fp32 + bias
    'dcn_offset_3x3_to_32_pair_direct_fp32': dict(
        N=3, sizes=[(25, 42)], cin=128, cout=32, k=3, bias=True, cout_real=18, out_dtype=torch.float32,
        expect=dict(pair=1, out_tma=0, n_tile=32)),
    # VIS sipmask_track: 768 -> 512 fp32 track features
    'vis_track_1x1_768_to_512_pair_direct_fp32': dict(
        N=3, sizes=[(25, 42)], cin=768, cout=512, k=1, bias=True, out_dtype=torch.float32,
        expect=dict(pair=1, out_tma=0, n_tiles_n=2)),
    # fp32 head outputs over five levels: fcos_cls|sip_cof (80 + 128), its 40-class VIS form (168 -> 176), fcos_reg|ctr (16)
    'head_multilevel_208_non_pair_direct_fp32': dict(
        N=3, sizes=LEVELS, cin=256, cout=208, k=3, bias=True, out_dtype=torch.float32, multi=True,
        expect=dict(pair=0, out_tma=0, n_tile=208)),
    'head_multilevel_176_non_pair_direct_fp32': dict(
        N=3, sizes=LEVELS, cin=256, cout=176, k=3, bias=True, cout_real=168, out_dtype=torch.float32, multi=True,
        expect=dict(pair=0, out_tma=0, n_tile=176)),
    'head_multilevel_16_alpha_non_pair_direct_fp32': dict(
        N=3, sizes=LEVELS, cin=256, cout=16, k=3, bias=True, cout_real=5, alpha=1.3, out_dtype=torch.float32, multi=True,
        expect=dict(pair=0, out_tma=0, n_tile=16)),
    # GN tower over five levels with an odd number of M tiles: the last pair has a dummy CTA
    'tower_gn_multilevel_odd_tiles_dummy_cta': dict(
        N=3, sizes=ODD_LEVELS, cin=256, cout=256, k=3, gn=True, multi=True,
        expect=dict(pair=1, out_tma=1, epi_split=0, tiles_m=45)),
    # 16-channel GroupNorm groups (Cout = 512) through the TMA-store epilogue
    'gn16_cout512_single_level_tma': dict(
        N=3, sizes=[(25, 42)], cin=256, cout=512, k=3, bias=True, gn=True, expect=dict(pair=1, out_tma=1, epi_split=0)),
    'gn16_cout512_multilevel_tma': dict(
        N=3, sizes=ODD_LEVELS, cin=256, cout=512, k=3, gn=True, multi=True, expect=dict(pair=1, out_tma=1, tiles_m=45)),
    # a single M tile: pair mode is refused although the N tile is a multiple of 32
    'single_m_tile_no_pair': dict(N=1, sizes=[(8, 16)], cin=256, cout=256, k=3, bias=True,
                                  expect=dict(pair=0, tiles_m=1, n_tile=64, out_tma=1)),
    # channel slices: input pitch 384 at channel 64, output pitch 320 at channel 32 (TMA store) ...
    'channel_slices_tma_fp16': dict(
        N=3, sizes=[(25, 42)], cin=256, cout=256, k=3, bias=True, relu=True, in_pitch=384, in_off=64, out_pitch=320,
        out_off=32, expect=dict(pair=1, out_tma=1)),
    # ... and fp32 direct stores into pitch 224 at channel 8
    'channel_slices_direct_fp32': dict(
        N=3, sizes=[(25, 42)], cin=256, cout=208, k=3, bias=True, in_pitch=320, in_off=64, out_pitch=224, out_off=8,
        out_dtype=torch.float32, expect=dict(pair=0, out_tma=0)),
    # a bias 4 bytes off 16-byte alignment: the split epilogue's float4 reads are impossible, smb_conv_run uses lockstep
    'split_plan_misaligned_bias_lockstep': dict(
        N=3, sizes=[(40, 56)], cin=64, cout=256, k=1, bias=True, bias_offset=1, residual='same', relu=True,
        expect=dict(TMA_SPLIT, res_tma=1)),
    'alpha_fp16_tma_lockstep': dict(N=3, sizes=[(25, 42)], cin=256, cout=256, k=3, bias=True, alpha=0.75, expect=TMA_SPLIT),
}


@pytest.fixture
def planner_defaults(monkeypatch):
    """Plans are created with the default planner knobs; the min_tiles knob is global state, restored afterwards."""
    from sipmask_b200 import conv
    for v in ('SMB_CONV_PAIR', 'SMB_CONV_SMALL', 'SMB_CONV_MIN_TILES', 'SMB_CONV_MAX_CTAS', 'SMB_CONV_CLUSTER',
              'SMB_CONV_EPI_SPLIT', 'SMB_CONV_STAGE_SETS', 'SMB_CONV_STORE_LAG', 'SMB_CONV_NO_TMA_STORE', 'SMB_CONV_NO_TMA_RES',
              'SMB_CONV_DEBUG'):
        monkeypatch.delenv(v, raising=False)
    prev = conv.set_min_tiles(0)
    yield
    conv.set_min_tiles(prev)


def _variants(case, info, monkeypatch):
    """(name, plan) pairs of the same convolution under different schedules."""
    from sipmask_b200 import conv

    def with_min_tiles(n, max_ctas=None):
        conv.set_min_tiles(n)
        try:
            p = case.new_plan()
        finally:
            conv.set_min_tiles(0)
        return p.set_max_ctas(max_ctas) if max_ctas else p

    def no_pair():
        monkeypatch.setenv('SMB_CONV_PAIR', '0')
        try:
            return case.new_plan()
        finally:
            monkeypatch.delenv('SMB_CONV_PAIR')

    yield 'one cluster walks every unit', case.new_plan().set_max_ctas(info['cluster'])
    yield 'grid capped at 7 CTAs', case.new_plan().set_max_ctas(7)
    yield 'widest N tile (min_tiles 1)', with_min_tiles(1)
    yield 'narrowest N tile (min_tiles 2^30)', with_min_tiles(1 << 30)
    yield 'serving tuning (min_tiles 16, 100 CTAs)', with_min_tiles(16, 100)
    yield 'SMB_CONV_PAIR=0', no_pair()


@pytest.mark.parametrize('name', sorted(CASES))
def test_plan_matches_fp64_reference_on_every_schedule(name, planner_defaults, monkeypatch):
    case = Case(name, **CASES[name])
    plan = case.new_plan()
    info = plan.info()
    for key, want in case.expect.items():
        assert info[key] == want, '%s: planner chose %s=%s, the case targets %s (plan %s)' % (name, key, info[key], want, info)
    if case.multi or case.stats:
        assert info['tiles_m'] == case.N * sum(_tiles(h, w) for h, w in case.out_sizes), info
    case.run(plan)
    bad = case.guard_problems(name)
    ratios = dict(out=_check_elements(case))
    if case.stats:
        ratios['stats'], bad_stats = _check_stats(case)
        bad += bad_stats
    assert not bad, '\n'.join(bad)
    ref = case.snapshot()
    case.run(plan)
    case.check_guards(name + ' (second run)')
    assert all(torch.equal(a, b) for a, b in zip(ref, case.snapshot())), '%s: a second run of the plan differs' % name
    for what, p in _variants(case, info, monkeypatch):
        case.run(p)
        case.check_guards('%s / %s' % (name, what))
        got = case.snapshot()
        for i, (a, b) in enumerate(zip(ref, got)):
            assert torch.equal(a, b), '%s / %s (plan %s): %s %d is not bit-identical to the default plan (%d elements differ)' % (
                name, what, p.info(), 'output' if i < len(case.outs) else 'stats', i, int((a != b).sum()))
    if case.stats:
        case.run(plan)
        ratios['gn_apply'] = _check_gn_apply(case)
    print('%s: worst err/bound %s plan %s' % (name, ' '.join('%s %.3g' % kv for kv in sorted(ratios.items())), info))


def test_misaligned_bias_matches_aligned_bias():
    """The lockstep epilogue a misaligned bias falls back to computes the split epilogue's values bit for bit."""
    spec = dict(CASES['split_plan_misaligned_bias_lockstep'])
    aligned = Case('split_plan_misaligned_bias_lockstep', **dict(spec, bias_offset=0))
    shifted = Case('split_plan_misaligned_bias_lockstep', **spec)
    assert aligned.bias.data_ptr() % 16 == 0 and shifted.bias.data_ptr() % 16 == 4
    assert torch.equal(aligned.bias, shifted.bias)
    out = []
    for case in (aligned, shifted):
        plan = case.new_plan()
        assert plan.info()['epi_split'] == 1
        case.run(plan)
        out.append(_bits(case.outs[0]))
    assert torch.equal(out[0], out[1])
