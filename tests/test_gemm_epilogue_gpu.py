"""The tensor-core GEMM's fused epilogue and side outputs, op by op against fp64 CPU references.

Every option the networks pass to a GEMM is exercised through cdx_op_gemm at the shapes of the real call sites in csrc/nets.cu
(conv3 / gn_silu_conv3, linear_into, the GEGLU projection, the fused q|k|v projection): bias, the per-sample row vector, the residual,
alpha, GEGLU, NCHW output, TF32 plane outputs (row-major and transposed), the channel-concat second source with its own range, and
the two side outputs later kernels trust: c_amax (the range the next fp16-split GEMM picks its exponent from) and c_stats (the
per-(image, channel) sums the next GroupNorm uses instead of a statistics pass).  Each case asserts the variant it ran (the plan
record: path, halo schedule, TMA or per-row epilogue, tile width, split-K, tail boxes) so that a planner change cannot silently move
a case off the variant it is meant to cover.  Modes: 1 = fp16 split (default), 3 = TF32 planes, 0 = FFMA tiles."""
import math
import os
import subprocess
import sys
import tempfile

import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

TOL = 2e-5
MODES = [1, 3, 0]
PATHS = {1: ('H16', 'H16_PAIR'), 3: ('TS',), 0: ('FFMA',)}
PLANS = []          # (case, plan) of every tensor-core case run in this process, printed at the end of the module


@pytest.fixture(scope='module')
def engines():
    from cycle_diffusion_b200.engine import Engine
    out = {}
    for m in MODES:
        out[m] = Engine(0)
        out[m].set_mma_mode(m)
    yield out
    print('\nplan records:')
    for case, plan in PLANS:
        print(f'  {case}: {plan}')


def rel(a, b):
    return float((a.double() - b.double()).abs().max() / max(1e-30, float(b.double().abs().max())))


def rn_tf32(x):
    """The kernels' rn_tf32 on fp32 values: add half a TF32 ulp to the bit pattern and clear the 13 low mantissa bits."""
    b = x.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    r = (b + 0x1000) & 0xFFFFE000
    return torch.where(r >= 2 ** 31, r - 2 ** 32, r).to(torch.int32).view(torch.float32)


def ref_gemm(x, w, bias=None, conv=None, x2=None, rowvec=None, rows_per_batch=1, residual=None, alpha=1.0, geglu=False):
    """fp64 CPU reference of the hook's C (dense rows [M, cols] or NHWC)."""
    xd, wd = x.double(), w.double()
    if conv is not None:
        s, p, up = conv.get('stride', 1), conv.get('pad', 1), conv.get('up', 1)
        xi = xd.permute(0, 3, 1, 2)
        if up > 1:
            xi = F.interpolate(xi, scale_factor=up, mode='nearest')
        y = F.conv2d(F.pad(xi, (0, 1, 0, 1)), wd, stride=2) if (s == 2 and p == 0) else F.conv2d(xi, wd, stride=s, padding=p)
        y = alpha * y.permute(0, 2, 3, 1)
        B = y.shape[0]
        y = y.reshape(-1, y.shape[-1])
    else:
        a = torch.cat([xd, x2.double()], 1) if x2 is not None else xd
        y = alpha * (a @ wd.t())
    if bias is not None:
        y = y + bias.double()
    if rowvec is not None:
        y = y + rowvec.double().repeat_interleave(rows_per_batch, 0)[:y.shape[0]]
    if residual is not None:
        y = y + residual.double().reshape(y.shape)
    if geglu:
        v, g = y.chunk(2, dim=1)
        y = v * F.gelu(g)
    return y.reshape(B, -1, y.shape[-1]) if conv is not None else y


def expect_plan(plan, mode, *, M, N, dense=True, out_nchw=False, tiles_m=None):
    """Invariants of the plan record that follow from the shape alone (the planner's tile width / split choice is pinned per case)."""
    assert plan['path'] in PATHS[mode], (mode, plan)
    if mode == 0:
        return
    h16 = mode == 1
    if tiles_m is not None and h16:
        assert (plan['path'] == 'H16_PAIR') == (tiles_m % 2 == 0), (tiles_m, plan)
    assert plan['epi_tma'] == int(h16 and dense and not out_nchw and plan['splits'] == 1 and M >= 128), plan
    tail = plan['epi_tma'] and ((plan['tn_w'] & 31) != 0 or ((N % plan['tn_w']) & 31) != 0)
    assert plan['tail16'] == int(bool(tail)), plan
    if plan['splits'] > 1:
        assert not plan['epi_tma'] and not (plan['side_done'] & 2), plan


def check_side_outputs(out, C, rows_per_batch, stats_tol=1e-5):
    """c_amax bit-equal to max |stored C|; c_stats against fp64 sums of the returned C."""
    if 'c_amax' in out:
        assert out['c_amax'].item() == C.abs().max().item(), (out['c_amax'].item(), C.abs().max().item())
    if 'c_stats' in out:
        Cd = C.double().reshape(-1, rows_per_batch, C.shape[-1])
        st = out['c_stats'].cpu()
        s_ref, q_ref = Cd.sum(1), (Cd * Cd).sum(1)
        assert float(((st[..., 0] - s_ref).abs() / Cd.abs().sum(1).clamp_min(1e-30)).max()) < stats_tol
        assert float(((st[..., 1] - q_ref).abs() / q_ref.clamp_min(1e-30)).max()) < stats_tol


def run_case(eng, mode, case, x, w, bias=None, *, repeat=True, **kw):
    """Run one GEMM on the GPU (twice for the tensor-core modes: bit-identical C and c_amax); returns (out dict, C on the CPU)."""
    dev = lambda t: t.cuda() if isinstance(t, torch.Tensor) else t
    args = {k: dev(v) for k, v in kw.items()}
    out = eng.op_gemm(dev(x), dev(w), dev(bias), **args)
    C = out['C'].cpu()
    if mode != 0:
        PLANS.append((f'mode {mode} {case}', out['plan']))
        if repeat:
            again = eng.op_gemm(dev(x), dev(w), dev(bias), **args)
            assert torch.equal(again['C'].cpu(), C), 'C differs between two identical calls'
            if 'c_amax' in out:
                assert torch.equal(again['c_amax'].cpu(), out['c_amax'].cpu())
            for k in ('C_lo', 'Ct_hi', 'Ct_lo'):
                if k in out:
                    assert torch.equal(again[k].cpu(), out[k].cpu())
    return out, C


def _gen(seed):
    return torch.Generator().manual_seed(seed)


# ---------------------------------------------------------------- residual / bias / row vector, dense
# (M, K, N, rows_per_batch): full 128-row tiles at the SD widths, ragged M (last tile on the per-row path), N with 16-column tail
# boxes (80, 112), N % 16 != 0 (per-row path), even / odd 128-row tile counts (CTA pair / single CTA), M < 128 (per-row launch)
DENSE = [(4096, 320, 320, 1024), (1024, 640, 640, 256), (1000, 320, 320, 1000), (1056, 320, 320, 352), (4096, 320, 80, 1024),
         (2048, 640, 112, 512), (4096, 320, 36, 1024), (1152, 640, 640, 384), (2048, 1280, 1280, 256), (100, 320, 640, 100)]


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('M,K,N,rpb', DENSE)
def test_dense_epilogue(engines, mode, M, K, N, rpb):
    g = _gen(M + K + N)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / math.sqrt(K)
    b = torch.randn(N, generator=g)
    rv = torch.randn(M // rpb, N, generator=g)
    res = torch.randn(M, N, generator=g) * 2
    alpha = 0.75
    out, C = run_case(engines[mode], mode, f'dense M{M} K{K} N{N}', x, w, b, rowvec=rv, rows_per_batch=rpb, residual=res, alpha=alpha,
                      c_amax=True, c_stats=True)
    ref = ref_gemm(x, w, b, rowvec=rv, rows_per_batch=rpb, residual=res, alpha=alpha)
    r = rel(C, ref)
    print(f'dense mode {mode} M{M} K{K} N{N}: rel {r:.2e} plan {out["plan"]}')
    assert r < TOL
    expect_plan(out['plan'], mode, M=M, N=N, tiles_m=-(-M // 128))
    if mode != 0:
        assert out['plan']['side_done'] & 1
        assert bool(out['plan']['side_done'] & 2) == (rpb % 32 == 0 and out['plan']['splits'] == 1)
    check_side_outputs(out, C, rpb)


# ---------------------------------------------------------------- conv3x3 (conv3 / gn_silu_conv3 shapes)
# (B, H, Cin, Cout, stride): 64x64 / 320 (halo, pair), 8x8 / 1280 at batch 8 (halo on pairs, two images per tile), ragged batches,
# an odd tile count (single CTA), a Downsample conv (stride 2) and a 16x16 / 640 level
CONV = [(1, 64, 320, 320, 1), (8, 8, 1280, 1280, 1), (3, 8, 320, 320, 1), (7, 8, 320, 320, 1), (5, 8, 320, 320, 1), (2, 32, 320, 320, 2),
        (2, 16, 640, 640, 1)]


def conv_tiles(B, H, stride):
    Ho = H // stride
    bw = min(Ho, 16)
    bh = min(Ho, 128 // bw)
    bn = 128 // (bw * bh)
    return (Ho // bw) * (Ho // bh) * -(-B // bn), bw, bh, bn


@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('B,H,Cin,Cout,stride', CONV)
def test_conv_epilogue(engines, mode, B, H, Cin, Cout, stride):
    g = _gen(B * 100 + H + Cin + Cout)
    x = torch.randn(B, H, H, Cin, generator=g)
    w = torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)
    b = torch.randn(Cout, generator=g)
    Ho = H // stride
    rv = torch.randn(B, Cout, generator=g)
    res = torch.randn(B, Ho, Ho, Cout, generator=g)
    conv = dict(stride=stride, pad=1, up=1)
    out, C = run_case(engines[mode], mode, f'conv B{B} {H}x{H} {Cin}->{Cout} s{stride}', x, w, b, conv=conv, rowvec=rv, residual=res,
                      c_amax=True, c_stats=True)
    ref = ref_gemm(x, w, b, conv=conv, rowvec=rv, rows_per_batch=Ho * Ho, residual=res)
    C = C.reshape(B, Ho * Ho, Cout)
    r = rel(C, ref)
    print(f'conv mode {mode} B{B} {H}x{H} {Cin}->{Cout} s{stride}: rel {r:.2e} plan {out["plan"]}')
    assert r < TOL
    tiles, bw, bh, bn = conv_tiles(B, H, stride)
    expect_plan(out['plan'], mode, M=B * Ho * Ho, N=Cout, dense=False, tiles_m=tiles)
    if mode == 1:
        pair = tiles % 2 == 0
        halo = stride == 1 and Cin % 64 == 0 and (bw + 2) * (bh + 2) * bn * 128 <= (25 if pair else 24) * 1024
        assert out['plan']['halo'] == int(halo), out['plan']
    check_side_outputs(out, C.reshape(-1, Cout), Ho * Ho)


# ---------------------------------------------------------------- GEGLU projection (value * exact-erf gelu(gate), bias)
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('M,K', [(4096, 320), (1000, 320), (1024, 640), (300, 1280)])
def test_geglu_epilogue(engines, mode, M, K):
    N = 8 * K
    g = _gen(M + K)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / math.sqrt(K)       # reference layout: [value rows; gate rows]
    b = torch.randn(N, generator=g) * 0.5
    out, C = run_case(engines[mode], mode, f'geglu M{M} K{K}', x, w, b, geglu=True, c_amax=True)
    ref = ref_gemm(x, w, b, geglu=True)
    r = rel(C, ref)
    print(f'geglu mode {mode} M{M} K{K}: rel {r:.2e} plan {out["plan"]}')
    assert C.shape == (M, N // 2) and r < TOL
    expect_plan(out['plan'], mode, M=M, N=N, tiles_m=-(-M // 128))
    check_side_outputs(out, C, M)


# ---------------------------------------------------------------- channel-concat second source with its own range
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('s1,s2', [(1e3, 1e-3), (1e-3, 1e3)])
def test_concat_sources_keep_their_ranges(engines, mode, s1, s2):
    """The decoder's skip concat as one GEMM over [x | x2]: both sources are scaled by the exponent of the larger of their two
    tracked ranges, so a source six orders of magnitude below the other still keeps the fp32 budget on its own contribution
    (measured on B200: a nine-order gap costs the small source ~3e-3, the limit of one shared exponent)."""
    M, C1, C2, N = 1024, 640, 320, 320
    g = _gen(7)
    x, x2 = torch.randn(M, C1, generator=g) * s1, torch.randn(M, C2, generator=g) * s2
    w = torch.randn(N, C1 + C2, generator=g) / math.sqrt(C1 + C2)
    b = torch.randn(N, generator=g) * s1
    out, C = run_case(engines[mode], mode, f'concat {s1:g}|{s2:g}', x, w, b, x2=x2, c_amax=True)
    assert rel(C, ref_gemm(x, w, b, x2=x2)) < TOL
    check_side_outputs(out, C, M)
    # the small source on its own: a weight that zeroes the large source's columns (the large source still runs through the GEMM)
    w0 = w.clone()
    if s1 > s2:
        w0[:, :C1] = 0
    else:
        w0[:, C1:] = 0
    out0, C0 = run_case(engines[mode], mode, f'concat {s1:g}|{s2:g} small source', x, w0, None, x2=x2)
    r = rel(C0, ref_gemm(x, w0, None, x2=x2))
    print(f'concat mode {mode} {s1:g} | {s2:g}: small source rel {r:.2e} plan {out0["plan"]}')
    assert r < TOL
    expect_plan(out0['plan'], mode, M=M, N=N, tiles_m=M // 128)
    if mode == 1:
        # a tracked range equal to the true max gives the same bits as the range measured by the GEMM
        am = torch.tensor([x.abs().max().item()]).cuda()
        am2 = torch.tensor([x2.abs().max().item()]).cuda()
        tr = engines[mode].op_gemm(x.cuda(), w0.cuda(), None, x2=x2.cuda(), a_amax=am, a2_amax=am2)['C'].cpu()
        assert torch.equal(tr, C0)


def test_tracked_range_matches_measured(engines):
    """a_amax equal to max |A| (dense and conv) gives bit-identical results to letting the GEMM measure it."""
    eng = engines[1]
    g = _gen(11)
    x = torch.randn(2048, 640, generator=g) * 3
    w = torch.randn(640, 640, generator=g) / 25
    am = torch.tensor([x.abs().max().item()]).cuda()
    assert torch.equal(eng.op_gemm(x.cuda(), w.cuda())['C'].cpu(), eng.op_gemm(x.cuda(), w.cuda(), a_amax=am)['C'].cpu())
    xc = torch.randn(2, 32, 32, 320, generator=g)
    wc = torch.randn(320, 320, 3, 3, generator=g) / 50
    amc = torch.tensor([xc.abs().max().item()]).cuda()
    conv = dict(stride=1, pad=1, up=1)
    assert torch.equal(eng.op_gemm(xc.cuda(), wc.cuda(), conv=conv)['C'].cpu(), eng.op_gemm(xc.cuda(), wc.cuda(), conv=conv, a_amax=amc)['C'].cpu())


# ---------------------------------------------------------------- split-K (small M, long K)
SPLITK = [(256, 2560, 320), (256, 5760, 640), (256, 11520, 1280), (256, 11520, 320)]


@pytest.mark.parametrize('mode', [1, 3])
@pytest.mark.parametrize('M,K,N', SPLITK)
def test_splitk_epilogue(engines, mode, M, K, N):
    rpb = 64
    g = _gen(M + K + N)
    x = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / math.sqrt(K)
    b = torch.randn(N, generator=g)
    rv = torch.randn(M // rpb, N, generator=g)
    res = torch.randn(M, N, generator=g)
    out, C = run_case(engines[mode], mode, f'splitk M{M} K{K} N{N}', x, w, b, rowvec=rv, rows_per_batch=rpb, residual=res, c_amax=True,
                      c_stats=True)
    r = rel(C, ref_gemm(x, w, b, rowvec=rv, rows_per_batch=rpb, residual=res))
    print(f'split-K mode {mode} M{M} K{K} N{N}: rel {r:.2e} plan {out["plan"]}')
    assert r < TOL
    assert out['plan']['splits'] > 1, out['plan']
    expect_plan(out['plan'], mode, M=M, N=N, tiles_m=M // 128)
    assert out['plan']['side_done'] == 1           # range from the reduce kernel, statistics from the extra pass
    check_side_outputs(out, C, rpb)


# ---------------------------------------------------------------- NCHW output (the final conv, N = 4)
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('B,H', [(2, 32), (3, 32)])
def test_nchw_output(engines, mode, B, H):
    Cin, Cout = 320, 4
    g = _gen(B + H)
    x = torch.randn(B, H, H, Cin, generator=g)
    w = torch.randn(Cout, Cin, 3, 3, generator=g) / math.sqrt(9 * Cin)
    b = torch.randn(Cout, generator=g)
    conv = dict(stride=1, pad=1, up=1)
    out, C = run_case(engines[mode], mode, f'nchw B{B} {H}x{H}', x, w, b, conv=conv, out_nchw=True)
    ref = ref_gemm(x, w, b, conv=conv).permute(0, 2, 1)          # [B, N, HW]
    r = rel(C, ref)
    print(f'nchw mode {mode} B{B}: rel {r:.2e} plan {out["plan"]}')
    assert C.shape == (B, Cout, H * H) and r < TOL
    expect_plan(out['plan'], mode, M=B * H * H, N=Cout, dense=False, out_nchw=True)


# ---------------------------------------------------------------- TF32 plane outputs (fused q|k|v projection)
@pytest.mark.parametrize('mode', [3, 1])
@pytest.mark.parametrize('M,Cc', [(4096, 320), (1000, 320), (1024, 640)])
def test_qkv_plane_outputs(engines, mode, M, Cc):
    N = 3 * Cc
    g = _gen(M + Cc)
    x = torch.randn(M, Cc, generator=g)
    w = torch.randn(N, Cc, generator=g) / math.sqrt(Cc)
    out, _ = run_case(engines[mode], mode, f'qkv planes M{M} C{Cc}', x, w, None, planes=True, t_col0=2 * Cc, c_amax=True)
    ref = ref_gemm(x, w)
    # the kernels' own fp32 result is hi + lo before rounding; lo must be rn_tf32(C - hi) of it, i.e. the rounding of the exact
    # fp32 difference: recover C as the fp32 value hi + lo rounds from and compare lo bit for bit with rn_tf32(C - hi)
    for hi, lo, r in ((out['C'].cpu(), out['C_lo'].cpu(), ref[:, :2 * Cc]), (out['Ct_hi'].cpu(), out['Ct_lo'].cpu(), ref[:, 2 * Cc:].t())):
        assert hi.shape == r.shape
        assert int((hi.view(torch.int32) & 0x1FFF).abs().max()) == 0, 'hi plane keeps mantissa bits below TF32'
        assert int((lo.view(torch.int32) & 0x1FFF).abs().max()) == 0, 'lo plane keeps mantissa bits below TF32'
        assert torch.equal(rn_tf32(hi), hi)
        # hi = rn_tf32(c) and lo = rn_tf32(c - hi) for the fp32 result c: |c - hi| <= half a TF32 ulp of hi, so lo is below it too
        ulp = torch.ldexp(torch.ones_like(hi), (torch.frexp(hi)[1] - 11).to(torch.int32))
        assert bool(((lo.abs() <= ulp / 2 * (1 + 2 ** -10)) | (hi == 0)).all()), 'lo larger than half a TF32 ulp of hi'
        err = float((hi.double() + lo.double() - r).abs().max() / r.abs().max())
        print(f'planes mode {mode} M{M} C{Cc}: rel {err:.2e}')
        assert err < TOL
    hi_all = torch.cat([out['C'].cpu().reshape(-1), out['Ct_hi'].cpu().reshape(-1)])
    assert out['c_amax'].item() == hi_all.abs().max().item()
    # lo == rn_tf32(C - hi) bit for bit, against the unsplit fp32 result of the same GEMM (same K split: same summation order)
    plain, Cp = run_case(engines[mode], mode, f'qkv plain M{M} C{Cc}', x, w, None, repeat=False)
    assert plain['plan']['splits'] == out['plan']['splits'] == 1, (plain['plan'], out['plan'])
    for hi, lo, c in ((out['C'].cpu(), out['C_lo'].cpu(), Cp[:, :2 * Cc]), (out['Ct_hi'].cpu(), out['Ct_lo'].cpu(), Cp[:, 2 * Cc:].t())):
        assert torch.equal(hi, rn_tf32(c))
        assert torch.equal(lo, rn_tf32(c - hi))


# ---------------------------------------------------------------- c_amax must not see rows / columns outside the tensor
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('case', ['dense M1000 N320', 'dense M1000 N36', 'conv B3 8x8'])
def test_amax_ignores_padding(engines, mode, case):
    """One column j has a zero weight row, a large bias (1000) and a residual that cancels half of it: every stored value of
    column j is 500 and every other output is O(1).  A range that takes padding rows (bias only) or padding columns into account
    reads 1000; one taken before the residual add reads 1000 too."""
    g = _gen(13)
    j = 5
    if case.startswith('dense'):
        M, N, K = 1000, int(case.split('N')[-1]), 320
        x = torch.randn(M, K, generator=g)
        w = torch.randn(N, K, generator=g) / math.sqrt(K)
        w[j] = 0
        res = torch.randn(M, N, generator=g) * 0.1
        conv, shape = None, (M, N)
    else:
        B, H, K, N = 3, 8, 320, 320
        x = torch.randn(B, H, H, K, generator=g)
        w = torch.randn(N, K, 3, 3, generator=g) / math.sqrt(9 * K)
        w[j] = 0
        res = torch.randn(B, H, H, N, generator=g) * 0.1
        conv, shape = dict(stride=1, pad=1, up=1), (B * H * H, N)
    b = torch.randn(N, generator=g) * 0.1
    b[j] = 1000.0
    res.view(-1, N)[:, j] = -500.0
    out, C = run_case(engines[mode], mode, f'padding {case}', x, w, b, conv=conv, residual=res, c_amax=True)
    C = C.reshape(shape)
    assert bool((C[:, j] == 500.0).all()) and float(C[:, torch.arange(N) != j].abs().max()) < 100
    assert out['c_amax'].item() == 500.0, out['c_amax'].item()


# ---------------------------------------------------------------- c_stats -> GroupNorm, against the statistics pass and fp64
@pytest.mark.parametrize('mode', MODES)
@pytest.mark.parametrize('kind', ['dense', 'conv'])
@pytest.mark.parametrize('ratio', [0, 30, 100])
def test_stats_feed_groupnorm(engines, mode, kind, ratio):
    """The epilogue's per-(image, channel) sums, fed to the GroupNorm, give the same normalised tensor as the GroupNorm's own fp64
    statistics pass -- also when a group's |mean| / std is 30 or 100 (E[x^2] - mean^2 cancels: fp32 partial sums of x and x^2 are
    not enough there)."""
    eng = engines[mode]
    g = _gen(17 + ratio)
    N = 320
    if kind == 'dense':
        B, HW, K = 4, 1024, 320
        x = torch.randn(B * HW, K, generator=g)
        w = torch.randn(N, K, generator=g) / math.sqrt(K)
        conv = None
    else:
        B, H, K = 2, 64, 320                   # (the 32 x 32 level takes split-K here: statistics by the extra pass)
        HW = H * H
        x = torch.randn(B, H, H, K, generator=g)
        w = torch.randn(N, K, 3, 3, generator=g) / math.sqrt(9 * K)
        conv = dict(stride=1, pad=1, up=1)
    b = ratio + 0.1 * torch.randn(N, generator=g)
    out, C = run_case(eng, mode, f'stats {kind} mean/std {ratio}', x, w, b, conv=conv, rows_per_batch=HW if conv is None else 0,
                      c_stats=True, repeat=False)
    C = C.reshape(B, HW, N)
    check_side_outputs(out, C.reshape(-1, N), HW)
    if mode != 0:
        assert out['plan']['side_done'] & 2, out['plan']           # the fused statistics are what is under test
    gamma = 1 + 0.1 * torch.randn(N, generator=g)
    beta = 0.1 * torch.randn(N, generator=g)
    ref = F.group_norm(C.double().permute(0, 2, 1), 32, gamma.double(), beta.double(), 1e-5).permute(0, 2, 1)
    xg = C.reshape(B, HW, 1, N).cuda()
    y_epi = eng.op_groupnorm(xg, gamma.cuda(), beta.cuda(), 1e-5, False, st1=out['c_stats']).cpu().reshape(B, HW, N)
    y_pass = eng.op_groupnorm(xg, gamma.cuda(), beta.cuda(), 1e-5, False).cpu().reshape(B, HW, N)
    r_epi, r_pass = rel(y_epi, ref), rel(y_pass, ref)
    print(f'stats {kind} mode {mode} mean/std {ratio}: GroupNorm rel err, epilogue statistics {r_epi:.2e}, statistics pass {r_pass:.2e}')
    assert r_pass < TOL and r_epi < TOL


# ---------------------------------------------------------------- GroupNorm hook: concat, scale-shift, caller statistics, amax
@pytest.mark.parametrize('C1,C2,B,HW', [(640, 320, 2, 256), (1280, 1280, 2, 64), (320, 0, 3, 1024)])
@pytest.mark.parametrize('scale_shift', [False, True])
def test_groupnorm_hook(engines, C1, C2, B, HW, scale_shift):
    eng = engines[1]
    g = _gen(C1 + C2 + HW)
    x = torch.randn(B, HW, C1, generator=g) * 3 + 1.5
    x2 = torch.randn(B, HW, C2, generator=g) * 0.5 - 2 if C2 else None
    Ct = C1 + C2
    gamma, beta = torch.randn(Ct, generator=g), torch.randn(Ct, generator=g)
    ss = torch.randn(B, 2 * Ct, generator=g) * 0.5 if scale_shift else None
    xc = torch.cat([x, x2], -1) if C2 else x
    ref = F.group_norm(xc.double().permute(0, 2, 1), 32, gamma.double(), beta.double(), 1e-6).permute(0, 2, 1)
    if scale_shift:
        ref = ref * (1 + ss[:, None, :Ct].double()) + ss[:, None, Ct:].double()
    ref = F.silu(ref)
    xd = x.reshape(B, HW, 1, C1).cuda()
    x2d = x2.reshape(B, HW, 1, C2).cuda() if C2 else None
    stats = lambda t: torch.stack([t.double().sum(1), (t.double() ** 2).sum(1)], -1)      # [B, C, 2] fp64
    for st1, st2 in ((None, None), (stats(x), stats(x2) if C2 else None)):
        y, am = eng.op_groupnorm(xd, gamma.cuda(), beta.cuda(), 1e-6, True, x2=x2d, scale_shift=ss.cuda() if ss is not None else None,
                                 st1=st1, st2=st2, amax=True)
        y = y.cpu().reshape(B, HW, Ct)
        r = rel(y, ref)
        print(f'groupnorm {C1}+{C2} B{B} HW{HW} ss={scale_shift} caller stats={st1 is not None}: rel {r:.2e}')
        assert r < TOL
        assert am.item() == y.abs().max().item()


# ---------------------------------------------------------------- the variants the tables above are meant to reach
def test_variant_coverage(engines):
    """Pinned shapes for each variant: TMA epilogue with a 16-column tail box, per-row epilogue (M < 128; TF32 path), split-K,
    CTA pair and single CTA, the conv3x3 halo schedule and the FFMA tiles."""
    def plan(mode, M, K, N, conv=None):
        g = _gen(M + K + N)
        if conv:
            x, w = torch.randn(conv[0], conv[1], conv[1], K, generator=g), torch.randn(N, K, 3, 3, generator=g) / math.sqrt(9 * K)
            return engines[mode].op_gemm(x.cuda(), w.cuda(), conv=dict(stride=1, pad=1, up=1))['plan']
        x, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / math.sqrt(K)
        return engines[mode].op_gemm(x.cuda(), w.cuda())['plan']
    p = plan(1, 4096, 320, 80)
    assert p['epi_tma'] and p['tail16'] and p['path'] == 'H16_PAIR', p
    p = plan(1, 100, 320, 640)
    assert not p['epi_tma'] and p['path'] == 'H16', p
    p = plan(3, 1000, 320, 36)
    assert not p['epi_tma'] and p['path'] == 'TS', p
    p = plan(1, 256, 11520, 320)
    assert p['splits'] > 1 and not p['epi_tma'], p
    p = plan(1, 1152, 640, 640)
    assert p['path'] == 'H16' and p['epi_tma'], p
    p = plan(1, 0, 320, 320, conv=(1, 64))
    assert p['halo'] and p['path'] == 'H16_PAIR', p
    p = plan(1, 0, 1280, 1280, conv=(8, 8))
    assert p['halo'] and p['path'] == 'H16_PAIR', p
    assert plan(0, 4096, 320, 320)['path'] == 'FFMA'


# ---------------------------------------------------------------- epilogue variants give the same bits
VARIANT_CASES = [('dense', 4096, 320, 320), ('dense', 4096, 320, 80), ('dense', 2048, 640, 112), ('dense', 1152, 640, 640),
                 ('geglu', 1024, 320, 2560), ('planes', 4096, 320, 640), ('conv', 1, 320, 320)]


def _variant_inputs(kind, M, K, N):
    g = _gen(M + K + N + 1)
    if kind == 'conv':
        x, w = torch.randn(1, 64, 64, K, generator=g), torch.randn(N, K, 3, 3, generator=g) / math.sqrt(9 * K)
        kw = dict(conv=dict(stride=1, pad=1, up=1), residual=torch.randn(1, 64, 64, N, generator=g), c_amax=True)
    else:
        x, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / math.sqrt(K)
        kw = dict(geglu=True, c_amax=True) if kind == 'geglu' else dict(planes=True, c_amax=True) if kind == 'planes' else \
            dict(residual=torch.randn(M, N, generator=g), rowvec=torch.randn(M // 128, N, generator=g), rows_per_batch=128, c_amax=True)
    return x, w, torch.randn(N, generator=g), kw


def _variant_outputs(path):
    """Run VARIANT_CASES on the default (fp16-split) engine and save the outputs (called in a fresh process per switch setting)."""
    from cycle_diffusion_b200.engine import Engine
    eng = Engine(0)
    res = {}
    for case in VARIANT_CASES:
        x, w, b, kw = _variant_inputs(*case)
        out = eng.op_gemm(x.cuda(), w.cuda(), b.cuda(), **{k: v.cuda() if isinstance(v, torch.Tensor) else v for k, v in kw.items()})
        res[case] = {k: (v.cpu() if isinstance(v, torch.Tensor) else v) for k, v in out.items()}
    torch.save(res, path)


def test_epilogue_switches_keep_results():
    """CDX_TC_NO_EPI_TMA=1 (every tile on the per-row epilogue) gives bit-identical C and c_amax: both epilogues do the same float
    operations in the same order.  CDX_TC_NO_PAIR=1 (single-CTA kernel only) stays within the fp32 budget."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    outs = {}
    with tempfile.TemporaryDirectory() as tmp:
        for flag in ('', 'CDX_TC_NO_EPI_TMA', 'CDX_TC_NO_PAIR'):
            env = {k: v for k, v in os.environ.items() if k not in ('CDX_TC_NO_EPI_TMA', 'CDX_TC_NO_PAIR')}
            if flag:
                env[flag] = '1'
            path = os.path.join(tmp, f'out{flag}.pt')
            code = f'import sys\nfrom tests.test_gemm_epilogue_gpu import _variant_outputs\n_variant_outputs({path!r})\n'
            r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True, cwd=root, env=env, timeout=600)
            assert r.returncode == 0, r.stderr[-2000:]
            outs[flag] = torch.load(path)
    base, no_tma, no_pair = outs[''], outs['CDX_TC_NO_EPI_TMA'], outs['CDX_TC_NO_PAIR']
    for case in VARIANT_CASES:
        kind, M, K, N = case
        x, w, b, kw = _variant_inputs(*case)
        print(f'{case}: default {base[case]["plan"]}  no-TMA {no_tma[case]["plan"]}  no-pair {no_pair[case]["plan"]}')
        assert not no_tma[case]['plan']['epi_tma'] and no_pair[case]['plan']['path'] == 'H16'
        if kind != 'conv':
            assert base[case]['plan']['epi_tma'], base[case]['plan']
        for k in base[case]:
            if k != 'plan':
                assert torch.equal(base[case][k], no_tma[case][k]), f'{case} {k}: TMA and per-row epilogues differ'
        ref = ref_gemm(x, w, b, conv=kw.get('conv'), rowvec=kw.get('rowvec'), rows_per_batch=kw.get('rows_per_batch', 1),
                       residual=kw.get('residual'), geglu=kw.get('geglu', False))
        got = no_pair[case]['C'].double() + (no_pair[case]['C_lo'].double() if 'C_lo' in no_pair[case] else 0)
        assert rel(got.reshape(ref.shape), ref) < TOL
        same = all(torch.equal(base[case][k], no_pair[case][k]) for k in base[case] if k != 'plan')
        print(f'  CTA pair vs single CTA: {"bit-identical" if same else "within tolerance, not bit-identical"}')
