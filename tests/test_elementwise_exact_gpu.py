"""Per-element conformance of the bf16 elementwise kernels that sit on every activation and gradient: BatchNorm apply
(+residual, ReLU), standalone ReLU forward / backward, axpby, 3x3/s2 max-pool, adaptive average pool, bilinear resize,
depthwise 3x3 convolution and the NHWC -> NCHW fp32 conversion.

Where the inputs can be built so that the fp32 arithmetic of the kernel is exact (integers, dyadic scale / shift, +-1
weights), the output must equal the correctly rounded (round-to-nearest-even) bf16 value of the float64 reference:
torch.equal.  Where it cannot (average pooling divides, bilinear weights are ATen's fp32 coordinate formulas), every
element must lie within one bf16 ulp OF THAT ELEMENT of RNE(float64 reference); the inputs are non-negative there, so no
cancellation makes an element's ulp meaningless.  Every kernel reads or writes a channel slice of a wider buffer (ld > C),
and the bytes outside the slice must stay untouched."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu

if torch.cuda.is_available():
    from seg_b200 import ops

DEV = "cuda"
CHANNELS = [48, 304, 2048]  # the 8-channel-vector kernels reject C % 8 != 0 (checked below with the decoder's 19)


def ints(shape, g, lo, hi):
    return torch.randint(lo, hi + 1, shape, generator=g).double()


def rne(t):
    """float64 -> bf16, rounded to nearest even.  Through float32 only where that step is exact (asserted)."""
    f = t.float()
    assert torch.equal(f.double(), t), "value not exact in fp32: the two-step rounding would not be RNE"
    return f.to(torch.bfloat16)


def rne64(t):
    """float64 -> bf16, round to nearest even, in one step: scale to an 8-bit significand, round half to even, scale back."""
    e = torch.floor(torch.log2(t.abs().clamp(min=2.0 ** -126)))
    q = torch.pow(2.0, e - 7)
    return (torch.round(t / q) * q).float().to(torch.bfloat16)  # exact: the rounded value has 9 significant bits at most


def ulp(b):
    """bf16 ulp of each element of a bf16 tensor (spacing to the next value away from zero)."""
    e = torch.floor(torch.log2(b.float().abs().clamp(min=2.0 ** -126)))
    return torch.pow(2.0, e - 7)


def assert_within_1ulp(name, got, ref64):
    want = rne64(ref64)
    g, w = got.float().cpu(), want.float()
    diff = (g - w).abs()
    bad = diff > ulp(want)
    if bad.any():
        idx = bad.nonzero()[:4]
        pytest.fail(f"{name}: {int(bad.sum())} elements more than 1 ulp from RNE(float64 reference); first {idx.tolist()}: "
                    f"got {[g[tuple(i)].item() for i in idx]} want {[w[tuple(i)].item() for i in idx]}")


def assert_exact(name, got, want):
    g = got.cpu()
    if not torch.equal(g, want):
        bad = (g.double() != want.double()).nonzero()[:4]
        pytest.fail(f"{name}: {int((g.double() != want.double()).sum())} elements differ from RNE(exact); first {bad.tolist()}: "
                    f"got {[g[tuple(i)].item() for i in bad]} want {[want[tuple(i)].item() for i in bad]}")


def sliced(vals, extra, off, fill=3.0):
    """vals [..., C] placed at channel offset `off` of a [..., C + extra] bf16 device buffer filled with `fill`."""
    buf = torch.full(vals.shape[:-1] + (vals.shape[-1] + extra,), fill, dtype=torch.bfloat16)
    buf[..., off:off + vals.shape[-1]] = rne(vals) if vals.dtype == torch.float64 else vals
    buf = buf.to(DEV)
    return buf, buf[..., off:off + vals.shape[-1]]


def assert_outside_untouched(name, buf, off, C, fill=3.0):
    b = buf.cpu().float()
    assert (b[..., :off] == fill).all() and (b[..., off + C:] == fill).all(), f"{name}: wrote outside its channel slice"


@pytest.mark.parametrize("C", CHANNELS)
def test_bn_apply_residual_relu_exact(C):
    g = torch.Generator().manual_seed(C)
    N, H, W = 2, 9, 11
    x = rne(ints((N, H, W, C), g, -300, 300)).double()  # bf16 values: the kernel reads exactly these
    res = rne(ints((N, H, W, C), g, -300, 300)).double()
    scale = ints((C,), g, -24, 24) / 8  # dyadic: x * scale + shift + res is exact in fp32
    shift = ints((C,), g, -400, 400) / 4
    ss = torch.cat([scale, shift]).float().to(DEV)
    xb, xv = sliced(x, 16, 8)
    rb, rv = sliced(res, 24, 16)
    ob, ov = sliced(torch.zeros(N, H, W, C, dtype=torch.float64), 8, 8)
    for relu in (True, False):
        ops.bn_apply(xv, ss, res=rv, out=ov, relu=relu)
        y = x * scale + shift + res
        assert_exact(f"bn_apply relu={relu} C={C}", ov, rne(y.clamp(min=0) if relu else y))
        assert_outside_untouched("bn_apply", ob, 8, C)
    ops.bn_apply(xv, ss, out=ov, relu=True)  # no residual
    assert_exact(f"bn_apply no-res C={C}", ov, rne((x * scale + shift).clamp(min=0)))
    # eval: scale / shift from running statistics (not dyadic): within one ulp of the float64 affine map of the returned ss
    gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    rm, rvar = torch.randn(C, generator=g), torch.rand(C, generator=g) + 0.5
    ss_e = ops.bn_eval_scale_shift(gamma.to(DEV), beta.to(DEV), rm.to(DEV), rvar.to(DEV), 1e-5)
    istd = 1.0 / torch.sqrt(rvar.double() + 1e-5)
    sc, sh = ss_e[:C].cpu().double(), ss_e[C:].cpu().double()
    assert torch.allclose(sc, gamma.double() * istd, rtol=2e-7, atol=0), "eval scale"
    assert torch.allclose(sh, beta.double() - rm.double() * gamma.double() * istd, rtol=1e-6, atol=1e-6), "eval shift"
    xs = x.abs() / 64  # exact bf16 values; non-negative so the affine map's relative error stays per element
    xb2, xv2 = sliced(xs, 16, 8)
    out = ops.bn_apply(xv2, ss_e, relu=False)
    ref = xs * sc + sh
    keep = ref.abs() > 1e-2 * ref.abs().max()  # away from the affine map's zero, where one ulp of the output is below fp32 noise
    assert_within_1ulp(f"bn_apply eval C={C}", out.cpu()[keep], ref[keep])


@pytest.mark.parametrize("C", CHANNELS)
def test_relu_axpby_exact(C):
    g = torch.Generator().manual_seed(100 + C)
    N, H, W = 2, 7, 13
    x = ints((N, H, W, C), g, -4000, 4000)
    _, xv = sliced(x, 8, 0)
    y = ops.relu_fwd(xv)
    assert_exact(f"relu_fwd C={C}", y, rne(rne(x).double().clamp(min=0)))
    xr = rne(x).double()
    dy = ints((N, H, W, C), g, -3000, 3000)
    old = ints((N, H, W, C), g, -3000, 3000)
    _, dyv = sliced(dy, 8, 8)
    _, yv2 = sliced(xr.clamp(min=0), 24, 16)
    db, dv = sliced(old, 8, 0)
    ops.relu_bwd(dyv, yv2, dv, 1.0)
    want = rne(torch.where(xr > 0, rne(dy).double(), 0.0) + rne(old).double())
    assert_exact(f"relu_bwd beta=1 C={C}", dv, want)
    assert_outside_untouched("relu_bwd", db, 0, C)
    for beta in (0.0, 1.0, 0.5, -2.0):
        a = ints((N, H, W, C), g, -3000, 3000)
        b = ints((N, H, W, C), g, -3000, 3000)
        _, av = sliced(a, 8, 8)
        bb, bv = sliced(b, 16, 8)
        ops.axpby(av, bv, beta)
        assert_exact(f"axpby beta={beta} C={C}", bv, rne(rne(a).double() + beta * rne(b).double()))
        assert_outside_untouched("axpby", bb, 8, C)


@pytest.mark.parametrize("C", CHANNELS)
def test_maxpool_exact_first_max(C):
    """ReLU zeros give ties: the kernel must pick ATen's first maximum, and the backward sums overlapping windows."""
    g = torch.Generator().manual_seed(200 + C)
    N, H, W = 2, 17, 19 if C < 2048 else 9
    x = ints((N, C, H, W), g, -6, 6).clamp(min=0).requires_grad_(True)
    y, idx_ref = F.max_pool2d(x, 3, 2, 1, return_indices=True)
    dy = ints(tuple(y.shape), g, -50, 50)
    y.backward(dy)
    yd, idx = ops.maxpool3x3s2_fwd(rne(x.detach().permute(0, 2, 3, 1).contiguous()).to(DEV))
    assert_exact(f"maxpool fwd C={C}", yd, rne(y.detach().permute(0, 2, 3, 1)))
    dx = ops.maxpool3x3s2_bwd(rne(dy.permute(0, 2, 3, 1).contiguous()).to(DEV), idx, (N, H, W, C))
    assert_exact(f"maxpool bwd C={C}", dx, rne(x.grad.permute(0, 2, 3, 1)))


@pytest.mark.parametrize("C", CHANNELS)
@pytest.mark.parametrize("bins", [1, 2, 3, 6])
def test_adaptive_avgpool_1ulp(bins, C):
    g = torch.Generator().manual_seed(300 + C + bins)
    N, H, W = 2, 33, 31
    x = ints((N, C, H, W), g, 0, 200).requires_grad_(True)
    y = F.adaptive_avg_pool2d(x, bins)
    dy = ints(tuple(y.shape), g, 0, 255)
    y.backward(dy)
    xb, xv = sliced(x.detach().permute(0, 2, 3, 1), 16, 8)
    yd = ops.adaptive_avgpool_fwd(xv, bins)
    assert_within_1ulp(f"avgpool fwd bins={bins} C={C}", yd, y.detach().permute(0, 2, 3, 1))
    old = ints((N, H, W, C), g, 0, 100)
    db, dv = sliced(old, 8, 8)
    ops.adaptive_avgpool_bwd(rne(dy.permute(0, 2, 3, 1).contiguous()).to(DEV), (N, H, W, C), bins, dx=dv, beta=1.0)
    assert_within_1ulp(f"avgpool bwd beta=1 bins={bins} C={C}", dv, x.grad.permute(0, 2, 3, 1) + old)
    assert_outside_untouched("avgpool bwd", db, 8, C)


@pytest.mark.parametrize("C", CHANNELS)
@pytest.mark.parametrize("ac", [True, False])
@pytest.mark.parametrize("sizes", [((9, 9), (33, 33)), ((33, 33), (129, 129)), ((8, 8), (31, 29)), ((33, 33), (17, 17))])
def test_bilinear_1ulp(sizes, ac, C):
    (Hi, Wi), (Ho, Wo) = sizes
    if C == 2048 and Ho > 64:
        pytest.skip("covered by the smaller maps at C = 2048")
    g = torch.Generator().manual_seed(400 + C)
    N = 2
    x = ints((N, C, Hi, Wi), g, 0, 255).requires_grad_(True)
    y = F.interpolate(x, size=(Ho, Wo), mode="bilinear", align_corners=ac)
    dy = ints(tuple(y.shape), g, 0, 255)
    y.backward(dy)
    _, xv = sliced(x.detach().permute(0, 2, 3, 1), 8, 0)
    ob, ov = sliced(torch.zeros(N, Ho, Wo, C, dtype=torch.float64), 16, 8)
    ops.bilinear_fwd(xv, Ho, Wo, ac, out=ov)
    assert_within_1ulp(f"bilinear fwd {sizes} ac={ac} C={C}", ov, y.detach().permute(0, 2, 3, 1))
    assert_outside_untouched("bilinear fwd", ob, 8, C)
    _, dyv = sliced(dy.permute(0, 2, 3, 1), 8, 8)
    old = ints((N, Hi, Wi, C), g, 0, 255)
    db, dv = sliced(old, 16, 0)
    ops.bilinear_bwd(dyv, Hi, Wi, ac, dx=dv, beta=1.0)
    assert_within_1ulp(f"bilinear bwd beta=1 {sizes} ac={ac} C={C}", dv, x.grad.permute(0, 2, 3, 1) + old)
    assert_outside_untouched("bilinear bwd", db, 0, C)


@pytest.mark.parametrize("C", CHANNELS)
@pytest.mark.parametrize("stride,dil", [(1, 1), (2, 1), (1, 2), (1, 4)])
def test_depthwise_exact(stride, dil, C):
    """SeparableConv2d.conv1: integer inputs and weights.  Wide-range data (outputs to ~+-4000) pins the bf16 rounding of
    the forward and of the beta = 1 data gradient, RNE(old + acc); small-range data (+-1 weights, |y| <= 36) pins the
    statistics, which are exact sums there."""
    g = torch.Generator().manual_seed(500 + C + 10 * stride + dil)
    N, H, W = 2, 17, 15
    pad = dil
    x = ints((N, C, H, W), g, -64, 64)
    w = ints((C, 1, 3, 3), g, -8, 8)
    y = F.conv2d(x, w, None, stride, pad, dil, groups=C)
    w9 = ops.dw_pack_weight(w.float().to(DEV))
    _, xv = sliced(x.permute(0, 2, 3, 1), 16, 8)
    ob, ov = sliced(torch.zeros(tuple(y.permute(0, 2, 3, 1).shape), dtype=torch.float64), 8, 0)
    ops.dwconv_fwd(xv, w9, stride, pad, dil, out=ov)
    assert_exact(f"dwconv fwd C={C}", ov, rne(y.permute(0, 2, 3, 1)))
    assert_outside_untouched("dwconv fwd", ob, 0, C)
    dy = ints(tuple(y.shape), g, -64, 64)
    acc = torch.nn.grad.conv2d_input(x.shape, w, dy, stride, pad, dil, groups=C).permute(0, 2, 3, 1)
    old = ints((N, H, W, C), g, -3000, 3000)
    db, dv = sliced(old, 16, 8)
    _, dyv = sliced(dy.permute(0, 2, 3, 1), 8, 8)
    ops.dwconv_bwd_data(dyv, w9, (N, H, W, C), stride, pad, dil, out=dv, beta=1.0)
    assert_exact(f"dwconv bwd_data beta=1 C={C}", dv, rne(rne(old).double() + acc))
    assert_outside_untouched("dwconv bwd_data", db, 8, C)
    gw = torch.nn.grad.conv2d_weight(x, w.shape, dy, stride, pad, dil, groups=C)
    g9 = ops.dwconv_bwd_weight(dyv, xv, stride, pad, dil)
    out = torch.empty(C, 1, 3, 3, device=DEV)
    ops.dw_unpack_wgrad(g9, out)
    assert_exact(f"dwconv bwd_weight C={C}", out, gw.float())
    # statistics of the output, exact: |y| <= 36
    xs = ints((N, C, H, W), g, -4, 4)
    ws = ints((C, 1, 3, 3), g, -1, 1)
    ys = F.conv2d(xs, ws, None, stride, pad, dil, groups=C).permute(0, 2, 3, 1).reshape(-1, C)
    stats = ops.new_stats(C, DEV)
    _, xsv = sliced(xs.permute(0, 2, 3, 1), 8, 8)
    ops.dwconv_fwd(xsv, ops.dw_pack_weight(ws.float().to(DEV)), stride, pad, dil, stats=stats)
    assert torch.equal(stats.cpu(), torch.cat([ys.sum(0), (ys * ys).sum(0)])), f"dwconv statistics C={C}"


@pytest.mark.parametrize("C", [19, 48, 304, 2048])
def test_nhwc_to_nchw_f32_exact(C):
    g = torch.Generator().manual_seed(600 + C)
    x = torch.randn(2, 9, 13, C, generator=g).to(torch.bfloat16)
    buf = torch.zeros(2, 9, 13, C + 5, dtype=torch.bfloat16)
    buf[..., 5:] = x
    y = ops.nhwc_to_nchw_f32(buf.to(DEV)[..., 5:])
    assert torch.equal(y.cpu(), x.float().permute(0, 3, 1, 2))


def test_vector_kernels_reject_unaligned_channels():
    """The 8-channel-vector kernels refuse C % 8 != 0 instead of computing on a partial vector."""
    x = torch.zeros(2, 5, 5, 19, dtype=torch.bfloat16, device=DEV)
    ss = torch.zeros(38, device=DEV)
    for fn in (lambda: ops.bn_apply(x, ss), lambda: ops.relu_fwd(x), lambda: ops.axpby(x, x.clone(), 1.0),
               lambda: ops.maxpool3x3s2_fwd(x), lambda: ops.adaptive_avgpool_fwd(x, 2), lambda: ops.bilinear_fwd(x, 9, 9, True)):
        with pytest.raises(RuntimeError):
            fn()
