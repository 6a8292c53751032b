"""Decode-head loss on bf16 / fp16 student logits (a decode head run under autocast).

The result must be what mmseg's `@force_fp32(apply_to=('seg_logit',))` losses compute on `seg_logit.float()`:
the loss and the accuracy of the fp32 path on the upcast logits, and a logits gradient of the logits' dtype equal
to (fp32 gradient * upstream gradient) rounded once. Every dispatch row of tests/test_gpu_weighted_ce.py is run
in both 16-bit dtypes and compared with the fp32 call on the upcast logits and with the float64 oracle."""
import pytest
import torch

from pfst_b200 import _lib, ops
from pfst_b200.losses import decode_head_losses, upsample_cross_entropy
from tests.test_gpu_weighted_ce import _DISPATCH, _case, _check_loss, _kernel_name, _oracle64, _view_at, UPSTREAM

pytestmark = pytest.mark.gpu
DTYPES = {"bf16": torch.bfloat16, "fp16": torch.float16}
TNAME = {torch.bfloat16: "__nv_bfloat16", torch.float16: "__half"}
LOSS_REL = 1e-7          # 16-bit vs fp32 on the upcast: the block sums meet in fp64 atomics in any order
# the fp32 gradient meets in float atomics (tile borders, shared-memory folds) in any order, so a rounded
# element may land one 16-bit ulp away; it may do so on at most this share of the elements
MAX_ULP_SHARE = 1e-3
# where the contributions to an element nearly cancel, the fp32 path's own reordering noise (a few fp32 ulps of
# the contributions) can exceed one 16-bit ulp of the small result: such an element may differ by more than one
# ulp, but by no more than this share of the gradient's largest magnitude
CANCEL_NOISE = 2.0 ** -20


def _ordered(t):
    """16-bit patterns as integers that are monotonic in the value (-0.0 and +0.0 both map to 0)."""
    i = t.contiguous().view(torch.int16).to(torch.int32)
    return torch.where(i < 0, -(i & 0x7fff), i)


def _check_grad16(got, want, what):
    """got, want: 16-bit gradients. NaN where the other is NaN; elsewhere at most one ulp apart, and bit-identical
    on all but a handful of elements."""
    assert got.dtype == want.dtype and got.shape == want.shape, (what, got.dtype, got.shape)
    nan_g, nan_w = torch.isnan(got), torch.isnan(want)
    assert torch.equal(nan_g, nan_w), (what, "NaN positions")
    ok = ~nan_w
    d = (_ordered(got) - _ordered(want)).abs()[ok]
    n_off = int((d != 0).sum())
    assert n_off <= max(4, int(MAX_ULP_SHARE * d.numel())), (what, n_off, d.numel())
    far = d > 1
    if far.any():
        g, w = got.float()[ok], want.float()[ok]
        scale = float(w[torch.isfinite(w)].abs().max())
        err = float((g - w)[far].abs().max())
        assert err <= CANCEL_NOISE * scale, (what, "ulps", int(d.max()), err, scale)


def _run_pair(z16, dl, dw, dcw=None, ignore_index=255, loss_weight=1.0, grad=True):
    """-> ((loss, acc, grad) of the 16-bit call, (loss, acc, grad rounded to the dtype) of the fp32 call on
    z16.float()), both with upstream gradient UPSTREAM when grad."""
    out = []
    for z in (z16, z16.float()):
        x = z.detach().clone().requires_grad_(grad)
        loss, acc = upsample_cross_entropy(x, dl, dw, dcw, ignore_index, loss_weight)
        if grad:
            (UPSTREAM * loss).backward()
        out.append((loss.detach(), acc, x.grad))
    (l16, a16, g16), (l32, a32, g32) = out
    assert l16.dtype == torch.float32 and a16.dtype == torch.float32
    if grad:
        assert g16.dtype == z16.dtype and g32.dtype == torch.float32
        g32 = g32.to(z16.dtype)
    return (l16, a16, g16), (l32, a32, g32)


def _check_pair(res16, res32, what):
    (l16, a16, g16), (l32, a32, g32) = res16, res32
    assert torch.equal(a16, a32), (what, float(a16), float(a32))
    lg, lw = float(l16), float(l32)
    assert abs(lg - lw) <= LOSS_REL * abs(lw), (what, lg, lw)
    if g16 is not None:
        _check_grad16(g16, g32, what)


def _row_inputs(kw, dtype, cuda, seed=5):
    logits, label, weight, _ = _case(2, kw["C"], 21, 37, kw.get("s", 4), seed=seed)
    z16 = logits.to(dtype)
    dl = _view_at(label.to(kw.get("dtype", torch.int64)), kw.get("lab_off", 0), cuda)
    dw = _view_at(weight, kw.get("w_off", 0), cuda)
    return z16, label, weight, dl, dw


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("row", range(len(_DISPATCH)), ids=[r[0].replace(" ", "") for r in _DISPATCH])
@pytest.mark.parametrize("grad", [True, False], ids=["grad", "nograd"])
def test_every_dispatch_row_matches_fp32_on_upcast_and_float64(cuda, dt, row, grad):
    what, kw, _ = _DISPATCH[row]
    dtype = DTYPES[dt]
    z16, label, weight, dl, dw = _row_inputs(kw, dtype, cuda)
    res16, res32 = _run_pair(z16.to(cuda), dl, dw, grad=grad)
    _check_pair(res16, res32, what)
    lo, _, _, _ = _oracle64(z16.float(), label, weight, None, 255, 1.0)
    _check_loss(res16[0], lo)


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("C,s", [(6, 4), (2, 4), (5, 4), (6, 2), (12, 4), (33, 4)])
def test_odd_offset_logits_views(cuda, dt, C, s):
    """A 16-bit view that starts one element into its storage (2-byte aligned) gives the same results."""
    dtype = DTYPES[dt]
    logits, label, weight, _ = _case(2, C, 21, 37, s, seed=60 + C)
    z16 = _view_at(logits.to(dtype), 1, cuda)
    assert z16.data_ptr() % 4 == 2
    res16, res32 = _run_pair(z16, label.to(cuda), weight.to(cuda))
    _check_pair(res16, res32, f"odd view C={C} x{s}")


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("C,s", [(6, 4), (5, 4), (6, 2), (12, 4)])
def test_options_match_fp32_on_upcast(cuda, dt, C, s):
    """Class weights, a loss weight != 1, ignore index -100 and uint8 labels on 16-bit logits."""
    dtype = DTYPES[dt]
    logits, label, weight, cw = _case(2, C, 21, 37, s, seed=7 * C + s, class_weight=True, ignore_index=-100)
    res16, res32 = _run_pair(logits.to(dtype).to(cuda), label.to(cuda), weight.to(cuda), cw.to(cuda), -100, 2.5)
    _check_pair(res16, res32, "options")
    logits, label, weight, cw = _case(2, C, 21, 37, s, seed=8 * C + s, class_weight=True)
    res16, res32 = _run_pair(logits.to(dtype).to(cuda), label.to(torch.uint8).to(cuda), weight.to(cuda),
                             cw.to(cuda), 255, 0.4)
    _check_pair(res16, res32, "options uint8")


@pytest.mark.parametrize("dt", list(DTYPES))
@pytest.mark.parametrize("C,s", [(6, 4), (5, 4), (6, 2), (33, 4)])
def test_non_finite_and_extreme_logits(cuda, dt, C, s):
    """+-inf and NaN logits (in one image) and, for fp16, logits near its largest finite value 65504: the NaN
    pattern and every value equal the fp32 path's on the upcast logits."""
    dtype = DTYPES[dt]
    logits, label, weight, _ = _case(2, C, 21, 37, s, seed=70 + C)
    z16 = logits.to(dtype)
    z16[0, 0, 3, 4] = float("inf")
    z16[0, 1 % C, 10, 30] = float("-inf")
    z16[0, C - 1, 17, 2] = float("nan")
    big = 65504.0 if dtype == torch.float16 else 2.0 ** 100
    z16[1, 0, 5:9, 20:26] = big
    z16[1, C - 1, 12:15, 3:8] = -big
    z16[1, 1 % C, 0, 0] = 0.5 * big
    res16, res32 = _run_pair(z16.to(cuda), label.to(cuda), weight.to(cuda))
    (l16, a16, g16), (l32, a32, g32) = res16, res32
    assert torch.equal(torch.isnan(l16), torch.isnan(l32)) and torch.equal(a16, a32)
    if not torch.isnan(l32):
        assert float(l16) == float(l32) or abs(float(l16) - float(l32)) <= LOSS_REL * abs(float(l32))
    _check_grad16(g16, g32, "non-finite")
    # the finite image alone: finite loss, gradient within one ulp
    res16, res32 = _run_pair(z16[1:].to(cuda), label[1:].to(cuda), weight[1:].to(cuda))
    assert torch.isfinite(res16[0]) and torch.isfinite(res32[0])
    _check_pair(res16, res32, "extreme finite")


def _scale_cast(src, scale, dst, tag):
    _lib.call("pfst_scale_cast", src.data_ptr(), scale.data_ptr(), src.numel(), dst.data_ptr(), tag, ops._stream())


def _cast_inputs():
    """Fixed fp32 inputs: normal values, fp16 / bf16 rounding ties, tiny and subnormal values, signed zeros,
    +-inf and NaN."""
    g = torch.Generator().manual_seed(11)
    parts = [torch.randn(4099, generator=g), 1e-3 * torch.randn(1001, generator=g),
             torch.tensor([1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8,
                           2.0 ** -24, 2.0 ** -25, 3 * 2.0 ** -26, 2.0 ** -14, 1e-40, -1e-40, 6e-39, 1.1e-38,
                           0.0, -0.0, -1e-30, 60000.0, 65519.0, 65520.0, -70000.0, 3.3e38, -3.4e38,
                           float("inf"), float("-inf"), float("nan")])]
    return torch.cat(parts)


@pytest.mark.parametrize("dt", ["fp32", "bf16", "fp16"])
@pytest.mark.parametrize("scale", [0.7, 1.0 / 3.0, 49152.0, 65536.0 * 0.7, 1e-5, -2.5])
@pytest.mark.parametrize("n", [0, 1, 3, 4, 5, 7, 1023, 5124])
def test_scale_cast_is_bit_exact(cuda, dt, scale, n):
    """pfst_scale_cast against torch's (g * s).to(dtype) on the device: one fp32 product, one rounding."""
    dtype = {"fp32": torch.float32, **DTYPES}[dt]
    g = _cast_inputs()
    g = torch.cat([g[-24:], g])[:n].to(cuda)                 # the special values first, so short calls see them
    s = torch.tensor(scale, dtype=torch.float32, device=cuda)
    want = (g * s).to(dtype)
    for src_off, dst_off in ((0, 0), (1, 1), (0, 1), (3, 2)):
        src = _view_at(g, src_off, cuda)
        dst = _view_at(torch.full((n,), 7.0, dtype=dtype), dst_off, cuda)
        _scale_cast(src, s, dst, ops._FLOAT2DT[dtype])
        nan = torch.isnan(want)
        assert torch.equal(torch.isnan(dst), nan), (src_off, dst_off)
        bits = torch.int32 if dtype == torch.float32 else torch.int16
        assert torch.equal(dst[~nan].view(bits), want[~nan].view(bits)), (src_off, dst_off)


def test_scale_cast_fp16_overflow_and_underflow(cuda):
    """A GradScaler-sized scale drives fp16 gradients to +-inf; a tiny one to subnormals and signed zeros."""
    g = torch.tensor([1.0, -1.0, 0.99, -2.0, 1e-4, 3e-6, -3e-6, 1e-12, -1e-12, 0.0], device=cuda)
    for scale, expect in ((65536.0, [float("inf"), float("-inf")]), (1.0, None)):
        s = torch.tensor(scale, device=cuda)
        dst = torch.empty(g.numel(), dtype=torch.float16, device=cuda)
        _scale_cast(g, s, dst, _lib.DT_F16)
        assert torch.equal(dst.view(torch.int16), (g * s).half().view(torch.int16))
        if expect:
            assert dst[0] == expect[0] and dst[1] == expect[1]
    dst = torch.empty(g.numel(), dtype=torch.float16, device=cuda)
    _scale_cast(g, torch.tensor(1.0, device=cuda), dst, _lib.DT_F16)
    assert 0 < float(dst[5]) < 2.0 ** -14                      # subnormal
    assert dst[8].view(torch.int16) == torch.tensor(-0.0, dtype=torch.float16).view(torch.int16)


def test_each_16bit_row_launches_the_twin_kernel_and_one_backward_kernel(cuda):
    from torch.profiler import ProfilerActivity, profile
    for dtype in DTYPES.values():
        for what, kw, want32 in _DISPATCH:
            z16, _, _, dl, dw = _row_inputs(kw, dtype, cuda)
            z = z16.to(cuda).requires_grad_(kw.get("grad", True))
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                loss, _ = upsample_cross_entropy(z, dl, dw)
                torch.cuda.synchronize()
            names = [_kernel_name(e.name) for e in prof.events() if "weighted_ce" in e.name]
            label_t = want32[want32.rindex(", ") + 2:-1]
            want = f"{want32[:want32.rindex(', ') + 2]}pfst::Lp<{label_t}, {TNAME[dtype]}>>"
            assert [n.replace(" ", "") for n in names] == [want.replace(" ", "")], (what, names, want)
            if not z.requires_grad:
                continue
            up = torch.full((), UPSTREAM, device=cuda)
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                torch.autograd.backward(loss, up)
                torch.cuda.synchronize()
            kernels = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
            assert len(kernels) == 1 and "scale_cast_kernel" in kernels[0], (what, kernels)
            assert z.grad.dtype == dtype


@pytest.mark.parametrize("dt,scaler_scale", [("bf16", None), ("fp16", 49152.0), ("fp16", 1.5e9)])
def test_autocast_conv_head_matches_float_path(cuda, dt, scaler_scale):
    """A small conv head under torch.autocast: handing its 16-bit logits to decode_head_losses gives the same
    logits gradient and, with a GradScaler, the same skip-or-step decision as the `.float()` path."""
    dtype = DTYPES[dt]
    g = torch.Generator().manual_seed(21)
    B, Cin, C, lh, lw = 2, 16, 6, 24, 40
    x = torch.randn((B, Cin, lh, lw), generator=g).to(cuda)
    label = torch.randint(0, C, (B, 1, 4 * lh, 4 * lw), generator=g)
    label[:, :, 5::9] = 255
    label = label.to(cuda)
    weight = torch.rand((B, 4 * lh, 4 * lw), generator=g).to(cuda)
    head0 = torch.nn.Conv2d(Cin, C, 3, padding=1).to(cuda)
    res = []
    for upcast in (False, True):
        head = torch.nn.Conv2d(Cin, C, 3, padding=1).to(cuda)
        head.load_state_dict(head0.state_dict())
        opt = torch.optim.SGD(head.parameters(), lr=0.1)
        scaler = torch.amp.GradScaler("cuda", init_scale=scaler_scale) if scaler_scale else None
        with torch.autocast("cuda", dtype=dtype):
            seg_logit = head(x)
            assert seg_logit.dtype == dtype
            seg_logit.retain_grad()
            out = decode_head_losses(seg_logit.float() if upcast else seg_logit, label, weight)
        loss = out["loss_ce"]
        (scaler.scale(loss) if scaler else loss).backward()
        stepped = None
        if scaler:
            before = [p.detach().clone() for p in head.parameters()]
            scaler.step(opt)
            scaler.update()
            stepped = not all(torch.equal(a, p) for a, p in zip(before, head.parameters()))
        else:
            opt.step()
        torch.cuda.synchronize()
        res.append((loss.detach(), out["acc_seg"], seg_logit.grad, stepped))
    (la, aa, ga, sa), (lb, ab, gb, sb) = res
    assert ga.dtype == dtype and gb.dtype == dtype
    assert torch.equal(aa, ab) and abs(float(la) - float(lb)) <= LOSS_REL * abs(float(lb))
    _check_grad16(ga, gb, "conv head")
    assert sa == sb
    if scaler_scale is not None:
        assert sa == (scaler_scale < 1e6), (scaler_scale, sa)           # 1.5e9 overflows fp16: skipped


def test_non_float_logits_raise_before_any_launch(cuda):
    from torch.profiler import ProfilerActivity, profile
    label = torch.zeros((1, 1, 32, 32), dtype=torch.int64, device=cuda)
    bad = [torch.zeros((1, 4, 8, 8), dtype=dt, device=cuda) for dt in (torch.float64, torch.int64, torch.int32,
                                                                        torch.uint8)]
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for z in bad:
            with pytest.raises(TypeError):
                upsample_cross_entropy(z, label)
            with pytest.raises(TypeError):
                decode_head_losses(z, label)
        torch.cuda.synchronize()
    assert not [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def test_unknown_tags_are_unsupported_even_with_null_pointers():
    lib = _lib.load()
    for tag in (-1, 3, 15, 19, 99):
        assert lib.pfst_weighted_ce_dt(None, tag, None, _lib.DT_I64, None, None, 1, 6, 8, 8, 32, 32, 255, 1.0,
                                       None, None, None, None) == -2
        assert lib.pfst_scale_cast(None, None, 16, None, tag, None) == -2
    # a known logit tag with an unknown label tag is refused the same way
    assert lib.pfst_weighted_ce_dt(None, _lib.DT_BF16, None, 7, None, None, 1, 6, 8, 8, 32, 32, 255, 1.0,
                                   None, None, None, None) == -2


@pytest.mark.parametrize("dt", list(DTYPES))
def test_empty_batch(cuda, dt):
    """B = 0: the reference's mean over no pixels (NaN) and accuracy 0; an empty gradient of the logits' dtype."""
    dtype = DTYPES[dt]
    logits, label, weight, _ = _case(0, 6, 8, 8, 4, seed=1)
    zl = logits.to(dtype).to(cuda).requires_grad_(True)
    loss, acc = upsample_cross_entropy(zl, label.to(cuda), weight.to(cuda))
    (UPSTREAM * loss).backward()
    assert torch.isnan(loss).item() and float(acc) == 0.0
    assert zl.grad.shape == logits.shape and zl.grad.dtype == dtype
    stats = torch.empty(4, dtype=torch.float64, device=cuda)
    out2 = torch.full((2,), 7.0, device=cuda)
    _lib.call("pfst_weighted_ce_dt", None, ops._FLOAT2DT[dtype], None, _lib.DT_I64, None, None, 0, 6, 8, 8, 32, 32,
              255, 1.0, None, stats.data_ptr(), out2.data_ptr(), ops._stream())
    res = out2.cpu()
    assert torch.isnan(res[0]) and float(res[1]) == 0.0, res
