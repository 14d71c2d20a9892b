"""GPU parity of the memory-bound kernels (BatchNorm fwd/bwd, MaxPool, PixelShuffle+blur+concat, cross-entropy,
optimizers, casts, weight staging, stitching) against the torch / numpy ops they replace.  Each test feeds both sides
the same bf16-rounded inputs, so tolerances are those of ONE op: 1e-2 (max-norm relative) for bf16 outputs, 1e-4..1e-3
for fp32 outputs, exact for integer / index results."""
import ctypes as C

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def rel(a, b):
    return ((a.float() - b.float()).abs().max() / b.float().abs().max().clamp_min(1e-20)).item()


def rnd(*shape, seed=0, scale=1.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return (torch.randn(*shape, generator=g, device="cuda") * scale).to(torch.bfloat16).float()


def nhwc(x, ld=None):
    from unet_b200.ops import padc
    n, c, h, w = x.shape
    ld = ld or padc(c)
    out = torch.zeros((n, h, w, ld), dtype=torch.bfloat16, device=x.device)
    out[..., :c] = x.permute(0, 2, 3, 1).to(torch.bfloat16)
    return out


def nchw(t, c):
    return t[..., :c].permute(0, 3, 1, 2).float()


def lib():
    from unet_b200 import _lib
    return _lib.load(), _lib


def S():
    return torch.cuda.current_stream().cuda_stream


def p(t):
    return None if t is None else t.data_ptr()


def f32(n, fill=0.0):
    return torch.full((n,), fill, dtype=torch.float32, device="cuda")


@pytest.mark.parametrize("N,Cc,H,W", [(4, 64, 32, 32), (2, 100, 17, 23), (3, 512, 8, 8)])
def test_bn_train_forward_backward(N, Cc, H, W):
    L, _lib = lib()
    from unet_b200.ops import padc, pad32
    x = (rnd(N, Cc, H, W, seed=1) * 2 + 0.5).to(torch.bfloat16).float()
    r = rnd(N, Cc, H, W, seed=2)
    gamma = (torch.rand(Cc, device="cuda") + 0.5)
    beta = torch.randn(Cc, device="cuda") * 0.1
    rm0, rv0 = torch.randn(Cc, device="cuda") * 0.1, torch.rand(Cc, device="cuda") + 0.5
    dz = rnd(N, Cc, H, W, seed=3)
    # torch reference: y = relu(bn(x) + r)
    xr = x.clone().requires_grad_(True)
    g_, b_ = gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)
    rm, rv = rm0.clone(), rv0.clone()
    y_pre = F.batch_norm(xr, rm, rv, g_, b_, True, 0.1, 1e-5) + r
    y_ref = F.relu(y_pre)

    ld, pix = padc(Cc), N * H * W
    xa, ra, dza = nhwc(x), nhwc(r), nhwc(dz)
    rows = 37
    part = torch.zeros((rows, 2, ld), dtype=torch.float32, device="cuda")
    _lib.check(L.b2u_bn_stats(p(xa), ld, pix, Cc, p(part), rows, ld, S()))
    mean, invstd, scale, shift = f32(pad32(Cc)), f32(pad32(Cc)), f32(pad32(Cc)), f32(pad32(Cc))
    rm2, rv2 = rm0.clone(), rv0.clone()
    scratch = torch.zeros(1 << 16, dtype=torch.float32, device="cuda")
    _lib.check(L.b2u_bn_finalize(p(part), rows, ld, Cc, float(pix), p(gamma), p(beta), 1e-5, 0.1, p(rm2), p(rv2),
                                 p(mean), p(invstd), p(scale), p(shift), p(scratch), scratch.numel(), S()))
    ya = torch.zeros_like(xa)
    _lib.check(L.b2u_bn_apply(p(xa), ld, p(scale), p(shift), p(ra), ld, None, None, 1, p(ya), ld, pix, Cc, S()))
    torch.cuda.synchronize()
    assert rel(nchw(ya, Cc), y_ref) <= 1e-2
    assert rel(rm2, rm) <= 1e-4 and rel(rv2, rv) <= 1e-4
    # backward with the (y > 0) mask of the block tail.  The reference uses the SAME mask (taken from the stored bf16
    # output): a pre-activation within rounding distance of 0 may flip sign between two fp32 evaluation orders, and one
    # flipped element would dominate a max-norm comparison without saying anything about the BN arithmetic.
    y_pre.backward(dz * (nchw(ya, Cc) > 0))
    part2 = torch.zeros((rows, 2, ld), dtype=torch.float32, device="cuda")
    _lib.check(L.b2u_bn_bwd_reduce(p(dza), ld, p(xa), ld, p(ya), ld, p(scale), p(shift), p(mean), p(invstd), 0, pix,
                                   Cc, p(part2), rows, ld, S()))
    dgamma, dbeta, mg, mgx = f32(Cc), f32(Cc), f32(pad32(Cc)), f32(pad32(Cc))
    _lib.check(L.b2u_bn_bwd_finalize(p(part2), rows, ld, Cc, float(pix), p(dgamma), p(dbeta), p(mg), p(mgx),
                                     p(scratch), scratch.numel(), S()))
    dxa = torch.zeros_like(xa)
    _lib.check(L.b2u_bn_bwd_apply(p(dza), ld, p(xa), ld, p(ya), ld, p(scale), p(shift), p(mean), p(invstd), p(gamma),
                                  p(mg), p(mgx), 0, 0, p(dxa), ld, pix, Cc, S()))
    torch.cuda.synchronize()
    assert rel(dgamma, g_.grad) <= 1e-3
    assert rel(dbeta, b_.grad) <= 1e-3
    assert rel(nchw(dxa, Cc), xr.grad) <= 1e-2
    # the single-launch variant (grid barrier inside) against torch and against the three-launch path; run twice to
    # check that the barrier words are left reusable
    sync = torch.zeros(2, dtype=torch.int32, device="cuda")
    for _ in range(2):
        dg2, db2, mg2, mgx2 = f32(Cc), f32(Cc), f32(pad32(Cc)), f32(pad32(Cc))
        dxf = torch.zeros_like(xa)
        part3 = torch.zeros((592, 2, ld), dtype=torch.float32, device="cuda")
        _lib.check(L.b2u_bn_bwd_fused(p(dza), ld, p(xa), ld, p(ya), ld, p(scale), p(shift), p(mean), p(invstd),
                                      p(gamma), 0, 0, p(dxf), ld, pix, Cc, p(part3), 592, ld, float(pix), p(dg2),
                                      p(db2), p(mg2), p(mgx2), p(sync), S()))
        torch.cuda.synchronize()
        assert rel(dg2, g_.grad) <= 1e-3 and rel(db2, b_.grad) <= 1e-3
        assert rel(dg2, dgamma) <= 1e-5 and rel(db2, dbeta) <= 1e-5
        assert rel(nchw(dxf, Cc), xr.grad) <= 1e-2
        assert rel(dxf, dxa) <= 1e-2 and (dxf[..., Cc:] == 0).all()
        assert sync[0].item() == 0


def test_bn_relu_mask_from_scale_shift_and_large_row_count():
    """conv->BN->ReLU backward: the mask is recomputed from x*scale+shift; also exercises the >128-row collapse."""
    L, _lib = lib()
    from unet_b200.ops import padc, pad32
    N, Cc, H, W = 8, 32, 64, 64
    x, dz = rnd(N, Cc, H, W, seed=1), rnd(N, Cc, H, W, seed=3)
    gamma, beta = torch.rand(Cc, device="cuda") + 0.5, torch.randn(Cc, device="cuda") * 0.1
    xr = x.clone().requires_grad_(True)
    y_pre = F.batch_norm(xr, None, None, gamma, beta, True, 0.1, 1e-5)
    ld, pix, rows = padc(Cc), N * H * W, 500
    xa, dza = nhwc(x), nhwc(dz)
    part = torch.zeros((rows, 2, ld), dtype=torch.float32, device="cuda")
    scratch = torch.zeros(1 << 16, dtype=torch.float32, device="cuda")
    mean, invstd, scale, shift, mg, mgx = (f32(pad32(Cc)) for _ in range(6))
    _lib.check(L.b2u_bn_stats(p(xa), ld, pix, Cc, p(part), rows, ld, S()))
    _lib.check(L.b2u_bn_finalize(p(part), rows, ld, Cc, float(pix), p(gamma), p(beta), 1e-5, 0.1, None, None, p(mean),
                                 p(invstd), p(scale), p(shift), p(scratch), scratch.numel(), S()))
    # same mask on both sides: sign of x*scale+shift evaluated exactly as the kernel does
    sc, sh = scale[:Cc].view(1, -1, 1, 1), shift[:Cc].view(1, -1, 1, 1)
    torch.cuda.synchronize()
    y_pre.backward(dz * ((x * sc + sh) > 0))
    assert ((y_pre > 0) != ((x * sc + sh) > 0)).float().mean().item() < 1e-4
    _lib.check(L.b2u_bn_bwd_reduce(p(dza), ld, p(xa), ld, None, 0, p(scale), p(shift), p(mean), p(invstd), 1, pix, Cc,
                                   p(part), rows, ld, S()))
    _lib.check(L.b2u_bn_bwd_finalize(p(part), rows, ld, Cc, float(pix), None, None, p(mg), p(mgx), p(scratch),
                                     scratch.numel(), S()))
    dxa = torch.zeros_like(xa)
    _lib.check(L.b2u_bn_bwd_apply(p(dza), ld, p(xa), ld, None, 0, p(scale), p(shift), p(mean), p(invstd), p(gamma),
                                  p(mg), p(mgx), 1, 0, p(dxa), ld, pix, Cc, S()))
    torch.cuda.synchronize()
    assert rel(nchw(dxa, Cc), xr.grad) <= 1e-2
    # fused single launch, accumulate mode (dx += ...), ReLU mask recomputed from scale/shift
    sync = torch.zeros(2, dtype=torch.int32, device="cuda")
    base = rnd(N, Cc, H, W, seed=9)
    dxf = nhwc(base)
    mg2, mgx2 = f32(pad32(Cc)), f32(pad32(Cc))
    part3 = torch.zeros((592, 2, ld), dtype=torch.float32, device="cuda")
    _lib.check(L.b2u_bn_bwd_fused(p(dza), ld, p(xa), ld, None, 0, p(scale), p(shift), p(mean), p(invstd), p(gamma),
                                  1, 1, p(dxf), ld, pix, Cc, p(part3), 592, ld, float(pix), None, None, p(mg2), p(mgx2),
                                  p(sync), S()))
    torch.cuda.synchronize()
    assert rel(nchw(dxf, Cc), xr.grad + base) <= 1e-2
    assert rel(mg2, mg) <= 1e-5 and rel(mgx2, mgx) <= 1e-5


@pytest.mark.parametrize("N,Cc,H,W", [(2, 64, 32, 32), (1, 24, 13, 9)])
def test_maxpool(N, Cc, H, W):
    L, _lib = lib()
    from unet_b200.ops import padc
    x = F.relu(rnd(N, Cc, H, W, seed=1))           # post-ReLU input: many exact ties at 0, as in the network
    x = (x * 4).round() / 4                          # and ties among positive values
    xr = x.clone().requires_grad_(True)
    y_ref = F.max_pool2d(xr, 3, 2, 1)
    dy = rnd(*y_ref.shape, seed=2)
    y_ref.backward(dy)
    ld = padc(Cc)
    xa, dya = nhwc(x), nhwc(dy)
    Ho, Wo = y_ref.shape[-2:]
    ya = torch.zeros((N, Ho, Wo, ld), dtype=torch.bfloat16, device="cuda")
    idx = torch.zeros((N, Ho, Wo, ld), dtype=torch.uint8, device="cuda")
    _lib.check(L.b2u_maxpool_fwd(p(xa), p(ya), p(idx), N, H, W, Cc, ld, S()))
    dxa = torch.full_like(xa, 1.0)
    _lib.check(L.b2u_maxpool_bwd(p(dya), p(idx), p(dxa), 1, N, H, W, Cc, ld, S()))   # accumulate onto ones
    torch.cuda.synchronize()
    assert torch.equal(nchw(ya, Cc), y_ref.detach())                                 # max of bf16 values: exact
    assert rel(nchw(dxa, Cc) - 1.0, xr.grad) <= 1e-2                                  # first-max tie rule as in ATen


@pytest.mark.parametrize("blur", [1, 0])
def test_shuffle_blur_concat_fwd_bwd(blur):
    L, _lib = lib()
    from unet_b200.layout import shuffle_row_of_co
    from unet_b200.ops import padc, pad32
    N, cu, cs, h, w = 2, 32, 24, 8, 12
    u = F.relu(rnd(N, 4 * cu, h, w, seed=1))          # conv1x1 output after ReLU, torch channel order (c,i,j)
    s = rnd(N, cs, 2 * h, 2 * w, seed=2)
    sscale, sshift = torch.rand(cs, device="cuda") + 0.5, torch.randn(cs, device="cuda") * 0.2
    ur, sr = u.clone().requires_grad_(True), s.clone().requires_grad_(True)
    up = F.pixel_shuffle(ur, 2)
    if blur:
        up = F.avg_pool2d(F.pad(up, (1, 0, 1, 0), mode="replicate"), 2, stride=1)
    cat_ref = F.relu(torch.cat([up, sr * sscale.view(1, -1, 1, 1) + sshift.view(1, -1, 1, 1)], 1))
    dcat = rnd(*cat_ref.shape, seed=3)
    # the plan stores d(cat) already masked by (cat > 0) (dgrad epilogue zmask); mimic that here
    cat_ref.backward(dcat)
    # kernel side: channels of u permuted to (i,j,c)
    roc = torch.tensor(shuffle_row_of_co(4 * cu), device="cuda")
    u_perm = torch.zeros_like(u)
    u_perm[:, roc] = u
    ua, sa = nhwc(u_perm), nhwc(s)
    ldc = padc(cu + cs)
    cat = torch.full((N, 2 * h, 2 * w, ldc), 3.0, dtype=torch.bfloat16, device="cuda")
    sc, sh = f32(pad32(cs)), f32(pad32(cs))
    sc[:cs], sh[:cs] = sscale, sshift
    _lib.check(L.b2u_shuffle_cat_fwd(p(ua), ua.shape[-1], cu, blur, p(sa), sa.shape[-1], cs, p(sc), p(sh), 1, p(cat),
                                     ldc, N, h, w, S()))
    torch.cuda.synchronize()
    assert rel(nchw(cat, cu + cs), cat_ref) <= 1e-2
    assert (cat[..., cu + cs:] == 0).all()
    # backward of the shuffle part
    dmasked = nhwc(dcat * (cat_ref > 0), ldc)
    du = torch.zeros_like(ua)
    _lib.check(L.b2u_shuffle_bwd(p(dmasked), ldc, p(ua), p(du), ua.shape[-1], cu, blur, N, h, w, S()))
    torch.cuda.synchronize()
    du_ref = (ur.grad * (u > 0))[:, :]            # (u > 0) mask of the conv1x1 ReLU is applied by the kernel
    got = torch.zeros_like(u)
    got[:] = nchw(du, 4 * cu)[:, roc]
    assert rel(got, du_ref) <= 1e-2


@pytest.mark.parametrize("Cc", [2, 8])
def test_cross_entropy(Cc):
    L, _lib = lib()
    N, H, W = 2, 32, 32
    P = N * H * W
    logits = torch.randn(P, 8 if Cc <= 8 else 16, device="cuda")
    labels = torch.randint(0, Cc, (P,), device="cuda", dtype=torch.uint8)
    w = torch.rand(Cc, device="cuda") + 0.1
    lr = logits[:, :Cc].clone().requires_grad_(True)
    ref = F.cross_entropy(lr, labels.long(), weight=w)
    ref.backward()
    rows = 64
    wp, lp = f32(rows), f32(rows)
    dl = torch.full((P, 16), 5.0, dtype=torch.bfloat16, device="cuda")
    loss = f32(1)
    _lib.check(L.b2u_ce_weight_sum(p(labels), P, p(w), Cc, p(wp), rows, S()))
    _lib.check(L.b2u_ce_fwd_bwd(p(logits), logits.shape[1], p(labels), P, Cc, p(w), p(wp), rows, p(dl), 16, p(lp),
                                rows, 1.0, S()))
    _lib.check(L.b2u_ce_finalize(p(lp), rows, p(wp), rows, p(loss), S()))
    torch.cuda.synchronize()
    assert abs(loss.item() - ref.item()) / abs(ref.item()) <= 1e-5
    assert rel(dl[:, :Cc], lr.grad) <= 1e-2
    assert (dl[:, Cc:] == 0).all()


def test_sgd_and_fastai_adam():
    from oracle.unet_oracle import fastai_adam_step
    L, _lib = lib()
    n = 10000
    p0, g = torch.randn(n, device="cuda"), torch.randn(n, device="cuda")
    pp = p0.clone()
    _lib.check(L.b2u_sgd_step(p(pp), p(g), n, 0.1, 0.5, S()))
    torch.cuda.synchronize()
    assert rel(pp, p0 - 0.1 * 0.5 * g) <= 1e-6
    # Adam: two segments with different lr / wd, three steps
    pa, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    pr, mr, vr = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    seg_end = torch.tensor([4000, n], dtype=torch.int64, device="cuda")
    seg_lr = torch.tensor([1e-3, 1e-2], device="cuda")
    seg_wd = torch.tensor([0.01, 0.0], device="cuda")
    for step in range(1, 4):
        gs = torch.randn(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(step))
        hyper = torch.tensor([0.9, 0.99, 1e-5, 1 - 0.9 ** step, 1 - 0.99 ** step, 1.0], device="cuda")
        _lib.check(L.b2u_adam_step(p(pa), p(gs), p(m), p(v), n, p(seg_end), p(seg_lr), p(seg_wd), 2, p(hyper), S()))
        fastai_adam_step(pr[:4000], gs[:4000], mr[:4000], vr[:4000], step, 1e-3, wd=0.01)
        fastai_adam_step(pr[4000:], gs[4000:], mr[4000:], vr[4000:], step, 1e-2, wd=0.0)
    torch.cuda.synchronize()
    assert rel(pa, pr) <= 1e-5


def test_layout_casts_and_crop():
    L, _lib = lib()
    N, Cc, H, W, ld = 2, 4, 16, 24, 16
    x8 = torch.randint(0, 256, (N, Cc, H, W), dtype=torch.uint8, device="cuda")
    y = torch.full((N, H, W, ld), 9.0, dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_nchw_to_nhwc(p(x8), 1, 255.0, 1.0, p(y), N, Cc, H, W, ld, 0, ld, S()))
    torch.cuda.synchronize()
    ref = (x8.float() / 255).to(torch.bfloat16)
    assert torch.equal(y[..., :Cc].permute(0, 3, 1, 2), ref) and (y[..., Cc:] == 0).all()
    xf = torch.rand((N, Cc, H, W), device="cuda")
    _lib.check(L.b2u_nchw_to_nhwc(p(xf), 0, 1.0, 1.0, p(y), N, Cc, H, W, ld, 0, ld, S()))
    back = torch.zeros((N, Cc, H, W), device="cuda")
    _lib.check(L.b2u_nhwc_to_nchw_f32(p(y), 0, ld, p(back), N, Cc, H, W, S()))
    torch.cuda.synchronize()
    assert torch.equal(back, xf.to(torch.bfloat16).float())
    # crop
    raster = torch.randint(0, 256, (Cc, 40, 50), dtype=torch.uint8, device="cuda")
    y0 = torch.tensor([0, 8, 24], dtype=torch.int32, device="cuda")
    x0 = torch.tensor([0, 34, 5], dtype=torch.int32, device="cuda")
    out = torch.zeros((3, 16, 16, ld), dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_crop_tiles(p(raster), 1, 255.0, 1.0, Cc, 40, 50, p(y0), p(x0), 3, 16, p(out), ld, S()))
    torch.cuda.synchronize()
    for t in range(3):
        ref = (raster[:, y0[t]:y0[t] + 16, x0[t]:x0[t] + 16].float() / 255).to(torch.bfloat16)
        assert torch.equal(out[t, ..., :Cc].permute(2, 0, 1), ref)


@pytest.mark.parametrize("dtype,code", [(torch.uint16, 2), (torch.int16, 3)])
def test_sixteen_bit_input_contract(dtype, code):
    """A0 for 16-bit imagery: bands are read as int32 -> float32 (data.py:24), the 'int16' batch transform divides by 255
    (utils.py:248-249, 288-289) and IntToFloatTensor by 255 again: two true fp32 divisions, then the bf16 cast.  The
    8-bit-valued case (max < 257: get_datatype says 'int8', utils.py:72-89) sees one division only.  Bit-exact."""
    L, _lib = lib()
    N, Cc, H, W, ld = 2, 4, 16, 24, 16
    g = torch.Generator().manual_seed(5)
    lo, hi = (0, 65536) if dtype == torch.uint16 else (-2000, 32768)
    xi = torch.randint(lo, hi, (N, Cc, H, W), generator=g, dtype=torch.int32)
    x = xi.to(dtype).cuda()
    y = torch.full((N, H, W, ld), 9.0, dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_nchw_to_nhwc(p(x), code, 255.0, 255.0, p(y), N, Cc, H, W, ld, 0, ld, S()))
    torch.cuda.synchronize()
    ref = xi.cuda().float().div_(255).div_(255).to(torch.bfloat16)       # the reference's two in-place divisions
    assert torch.equal(y[..., :Cc].permute(0, 3, 1, 2), ref) and (y[..., Cc:] == 0).all()
    _lib.check(L.b2u_nchw_to_nhwc(p(x), code, 255.0, 1.0, p(y), N, Cc, H, W, ld, 0, ld, S()))
    torch.cuda.synchronize()
    assert torch.equal(y[..., :Cc].permute(0, 3, 1, 2), (xi.cuda().float() / 255).to(torch.bfloat16))
    # crop from a 16-bit raster
    ri = torch.randint(lo, hi, (Cc, 40, 50), generator=g, dtype=torch.int32)
    raster = ri.to(dtype).cuda()
    y0 = torch.tensor([0, 8, 24], dtype=torch.int32, device="cuda")
    x0 = torch.tensor([0, 34, 5], dtype=torch.int32, device="cuda")
    out = torch.zeros((3, 16, 16, ld), dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_crop_tiles(p(raster), code, 255.0, 255.0, Cc, 40, 50, p(y0), p(x0), 3, 16, p(out), ld, S()))
    torch.cuda.synchronize()
    for t in range(3):
        ref = ri[:, y0[t]:y0[t] + 16, x0[t]:x0[t] + 16].cuda().float().div_(255).div_(255).to(torch.bfloat16)
        assert torch.equal(out[t, ..., :Cc].permute(2, 0, 1), ref)
    with pytest.raises(_lib.B2UError):
        _lib.check(L.b2u_nchw_to_nhwc(p(x), 7, 255.0, 1.0, p(y), N, Cc, H, W, ld, 0, ld, S()))


def test_mse_loss_and_regression_sums():
    """MSELossFlat(axis=1) fwd + bwd (train.py:189-192) against torch, and the sums behind fastai's rmse / R2Score."""
    L, _lib = lib()
    P_, ld, ldg, rows = 3 * 40 * 56, 8, 16, 37
    g = torch.Generator(device="cuda").manual_seed(2)
    pred = torch.randn((P_, ld), device="cuda", generator=g) * 3
    tgt = torch.randn(P_, device="cuda", generator=g) * 2 + 1
    dp = torch.full((P_, ldg), 7.0, dtype=torch.bfloat16, device="cuda")
    part = torch.zeros(rows, device="cuda")
    loss = torch.zeros(1, device="cuda")
    _lib.check(L.b2u_mse_fwd_bwd(p(pred), ld, p(tgt), P_, p(dp), ldg, p(part), rows, 1.0, S()))
    _lib.check(L.b2u_mse_finalize(p(part), rows, P_, p(loss), S()))
    torch.cuda.synchronize()
    z = pred[:, 0].clone().requires_grad_(True)
    ref = torch.nn.functional.mse_loss(z, tgt)
    ref.backward()
    assert abs(loss.item() - ref.item()) <= 1e-5 * abs(ref.item())
    assert rel(dp[:, 0].float(), z.grad) <= 2.0 ** -8 and (dp[:, 1:] == 0).all()
    sums = torch.zeros(4, dtype=torch.float64, device="cuda")
    partial = torch.zeros(rows * 3, dtype=torch.float64, device="cuda")
    ticket = torch.zeros(1, dtype=torch.int32, device="cuda")
    for _ in range(2):       # two validation batches accumulate
        _lib.check(L.b2u_regression_sums(p(pred), ld, p(tgt), P_, p(partial), rows, p(sums), p(ticket), S()))
    torch.cuda.synchronize()
    d = (pred[:, 0].double() - tgt.double())
    want = torch.stack([2 * (d * d).sum(), 2 * tgt.double().sum(), 2 * (tgt.double() ** 2).sum(),
                        torch.tensor(2.0 * P_, dtype=torch.float64, device="cuda")])
    assert torch.allclose(sums, want, rtol=1e-12)


@pytest.mark.parametrize("C", [2, 8, 13])
def test_dice_counts(C):
    """DiceMulti counts (train.py:196) against the oracle's dice_multi: exact integers."""
    from oracle.unet_oracle import dice_multi
    L, _lib = lib()
    P_, ld = 5 * 33 * 47, 8 if C <= 8 else 16
    g = torch.Generator(device="cuda").manual_seed(C)
    logits = torch.randn((P_, ld), device="cuda", generator=g)
    logits[::7, 1] = logits[::7, 0]          # ties: the first maximum wins, as torch.argmax
    labels = torch.randint(0, C, (P_,), device="cuda", generator=g, dtype=torch.int64).to(torch.uint8)
    counts = torch.zeros(3 * C, dtype=torch.int64, device="cuda")
    _lib.check(L.b2u_dice_counts(p(logits), ld, p(labels), P_, C, p(counts), S()))
    _lib.check(L.b2u_dice_counts(p(logits), ld, p(labels), P_, C, p(counts), S()))    # accumulates over batches
    torch.cuda.synchronize()
    pred = logits[:, :C].argmax(1)
    for c in range(C):
        assert counts[c].item() == 2 * ((pred == c) & (labels == c)).sum().item()
        assert counts[C + c].item() == 2 * (pred == c).sum().item()
        assert counts[2 * C + c].item() == 2 * (labels == c).sum().item()
    inter, ps, ts = counts[:C].double(), counts[C:2 * C].double(), counts[2 * C:].double()
    dice = [(2 * inter[c] / (ps[c] + ts[c])).item() for c in range(C) if ps[c] + ts[c] > 0]
    assert abs(sum(dice) / len(dice) - dice_multi(pred, labels.long(), C)) <= 1e-12


def test_regression_stitch_mode2():
    """regression merge (predict.py:300-316) through `b2u_stitch_accumulate` mode 2 with the tile count on the device:
    raw predictions summed, divided by the count, -9999 where no tile was placed - against the numpy restatement of
    the reference's merge."""
    from oracle.stitch import merge_pixel_windows_regression
    L, _lib = lib()
    T, P_, ld, Y, X = 6, 16, 8, 40, 52
    g = torch.Generator(device="cuda").manual_seed(9)
    z = torch.randn((T, P_, P_, ld), device="cuda", generator=g)
    wins = [(0, 0, P_, P_), (12, 0, P_, P_), (24, 0, P_, P_), (0, 12, P_, P_), (12, 12, P_, P_), (30, 20, P_, P_)]
    from unet_b200.tiling import colour_classes
    y0 = torch.tensor([w[1] for w in wins], dtype=torch.int32, device="cuda")
    x0 = torch.tensor([w[0] for w in wins], dtype=torch.int32, device="cuda")
    acc = torch.zeros((1, Y, X), device="cuda")
    cnt = torch.zeros((Y, X), dtype=torch.uint8, device="cuda")
    for cls in colour_classes(wins):
        sel = torch.tensor(cls, dtype=torch.int32, device="cuda")
        n_sel = torch.tensor([len(cls)], dtype=torch.int32, device="cuda")
        _lib.check(L.b2u_stitch_accumulate(p(z), ld, 1, T, P_, P_, p(y0), p(x0), p(sel), p(n_sel), len(cls), 2, p(acc),
                                           p(cnt), Y, X, 0, 0, S()))
    out = torch.zeros((1, Y, X), device="cuda")
    _lib.check(L.b2u_stitch_finalize_mean(p(acc), p(cnt), 1, Y, X, -9999.0, p(out), S()))
    torch.cuda.synchronize()
    ref = merge_pixel_windows_regression([z[t, :, :, 0].cpu().numpy()[None] for t in range(T)], wins, Y, X)
    import numpy as np
    got = out[0].cpu().numpy()
    assert (got == -9999).sum() == (ref == -9999).sum() > 0
    assert np.allclose(got, ref, rtol=1e-6, atol=1e-6)


@pytest.mark.parametrize("Cout,Cin,ks", [(16, 12, 3), (100, 100, 3), (384, 96, 1), (40, 4, 3)])
def test_stage_weights(Cout, Cin, ks):
    L, _lib = lib()
    from unet_b200.layout import shuffle_row_of_co
    from unet_b200.ops import padc, pad32
    kk = ks * ks
    w = torch.randn(Cout, Cin, ks, ks, device="cuda")
    b = torch.randn(Cout, device="cuda")
    roc = torch.tensor(shuffle_row_of_co(Cout), dtype=torch.int32, device="cuda")
    wf = torch.zeros((Cout, kk, padc(Cin)), dtype=torch.bfloat16, device="cuda")
    wd = torch.zeros((Cin, kk, padc(Cout)), dtype=torch.bfloat16, device="cuda")
    br = f32(pad32(Cout))
    it = _lib.WStageItem()
    it.w, it.bias, it.row_of_co, it.wf, it.wd, it.bias_rows = p(w), p(b), p(roc), p(wf), p(wd), p(br)
    it.Cout, it.Cin, it.kk, it.wf_cinp, it.wd_coutp, it.scale, it.block_start = Cout, Cin, kk, padc(Cin), padc(Cout), 0.25, 0
    dev_items = torch.frombuffer(bytearray(bytes(it)), dtype=torch.uint8).cuda()
    _lib.check(L.b2u_stage_weights(p(dev_items), 1, ((Cout + 31) // 32) * ((Cin + 31) // 32), S()))
    torch.cuda.synchronize()
    ws = (w * 0.25).to(torch.bfloat16)
    ref_f = torch.zeros_like(wf)
    ref_f[roc.long(), :, :Cin] = ws.permute(0, 2, 3, 1).reshape(Cout, kk, Cin)
    ref_d = torch.zeros_like(wd)
    ref_d[:, :, roc.long()] = ws.flip(2, 3).permute(1, 2, 3, 0).reshape(Cin, kk, Cout)
    assert torch.equal(wf, ref_f) and torch.equal(wd, ref_d)
    ref_b = torch.zeros_like(br)
    ref_b[roc.long()] = b
    assert torch.equal(br, ref_b)


@pytest.mark.parametrize("H,W,P,ov,Cc", [(300, 420, 64, 0.125, 2), (257, 511, 128, 0.5, 3)])
def test_stitch_mode0_against_numpy_merge(H, W, P, ov, Cc):
    """softmax + overlap accumulate (`b2u_stitch_accumulate` mode 0, tile count on the device) + normalise + argmax vs
    the numpy restatement of predict.py:284-337."""
    from oracle.stitch import merge_pixel_windows, softmax_probs
    from unet_b200.tiling import colour_classes, compute_windows
    L, _lib = lib()
    wins = compute_windows(H, W, P, ov)
    T = len(wins)
    g = torch.Generator(device="cuda").manual_seed(5)
    logits = torch.randn((T, P, P, 8), generator=g, device="cuda") * 3
    probs = [softmax_probs(logits[t, ..., :Cc].permute(2, 0, 1).cpu().numpy()) for t in range(T)]
    ref = merge_pixel_windows(probs, wins, H, W)
    acc = torch.zeros((Cc, H, W), dtype=torch.float32, device="cuda")
    cnt = torch.zeros((H, W), dtype=torch.uint8, device="cuda")
    mask = torch.zeros((H, W), dtype=torch.uint8, device="cuda")
    y0 = torch.tensor([w[1] for w in wins], dtype=torch.int32, device="cuda")
    x0 = torch.tensor([w[0] for w in wins], dtype=torch.int32, device="cuda")
    for cls in colour_classes(wins):
        sel = torch.tensor(cls, dtype=torch.int32, device="cuda")
        n_sel = torch.tensor([len(cls)], dtype=torch.int32, device="cuda")
        _lib.check(L.b2u_stitch_accumulate(p(logits), 8, Cc, T, P, P, p(y0), p(x0), p(sel), p(n_sel), len(cls), 0,
                                           p(acc), p(cnt), H, W, 0, 0, S()))
    _lib.check(L.b2u_stitch_finalize(p(acc), p(cnt), Cc, H, W, 0, p(mask), S()))
    torch.cuda.synchronize()
    # coverage counts are integers: exact;  the class mask agrees except where two class means tie within fp32 rounding
    cov = np.zeros((H, W), np.int64)
    for (x, y, w, h) in wins:
        cov[y:y + h, x:x + w] += 1
    assert np.array_equal(cnt.cpu().numpy().astype(np.int64), cov)
    agree = (mask.cpu().numpy() == ref).mean()
    assert agree >= 0.9999, agree


def test_pointwise_smallk_head_dgrad():
    L, _lib = lib()
    from unet_b200.ops import padc
    P, Cc, K = 5000, 100, 2
    dl = rnd(P, K, seed=1)
    w = rnd(K, Cc, seed=2)                     # torch head weight [n_out][C]
    zz = rnd(P, Cc, seed=3)
    ref = (dl @ w) * (zz > 0)
    a = torch.zeros((P, 16), dtype=torch.bfloat16, device="cuda"); a[:, :K] = dl.to(torch.bfloat16)
    wd = torch.zeros((Cc, 16), dtype=torch.bfloat16, device="cuda"); wd[:, :K] = w.t().to(torch.bfloat16)
    ld = padc(Cc)
    z = torch.zeros((P, ld), dtype=torch.bfloat16, device="cuda"); z[:, :Cc] = zz.to(torch.bfloat16)
    out = torch.full((P, ld), 3.0, dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_pointwise_smallk(p(a), 16, K, p(wd), 16, p(z), ld, p(out), ld, P, Cc, S()))
    torch.cuda.synchronize()
    assert rel(out[:, :Cc], ref) <= 1e-2
    assert (out[:, Cc:] == 0).all()


@pytest.mark.parametrize("n,C", [(256, 48), (1024, 384), (625, 40), (64, 384)])
def test_softmax_dim1_transposes_and_batched_transpose(n, C):
    """softmax over the QUERY axis with its transposed copy (fastai SelfAttention: F.softmax(bmm(f^T, g), dim=1)), its
    backward with the transposed dS, and the batched [n, C] -> [C, n] transpose that puts contraction indices innermost."""
    from unet_b200.ops import padc
    L, _lib = lib()
    B, ld = 3, padc(n)
    g = torch.Generator(device="cuda").manual_seed(n)
    Sm = torch.zeros((B, n, ld), dtype=torch.bfloat16, device="cuda")
    Sm[..., :n] = (torch.randn((B, n, n), device="cuda", generator=g) * 2).to(torch.bfloat16)
    beta, betaT = torch.zeros_like(Sm), torch.zeros_like(Sm)
    _lib.check(L.b2u_softmax_dim1(p(Sm), p(beta), p(betaT), B, n, ld, S()))
    torch.cuda.synchronize()
    ref = torch.softmax(Sm[..., :n].float(), dim=1)
    assert rel(beta[..., :n], ref) <= 2.0 ** -8
    assert torch.equal(betaT[..., :n], beta[..., :n].transpose(1, 2))
    db = torch.zeros_like(Sm)
    db[..., :n] = torch.randn((B, n, n), device="cuda", generator=g).to(torch.bfloat16)
    dS, dST = torch.zeros_like(Sm), torch.zeros_like(Sm)
    _lib.check(L.b2u_softmax_dim1_bwd(p(beta), p(db), p(dS), p(dST), B, n, ld, S()))
    torch.cuda.synchronize()
    bf, dbf = beta[..., :n].float(), db[..., :n].float()
    ref_ds = bf * (dbf - (bf * dbf).sum(1, keepdim=True))
    assert rel(dS[..., :n], ref_ds) <= 1e-2
    assert torch.equal(dST[..., :n], dS[..., :n].transpose(1, 2))
    x = torch.zeros((B, n, padc(C)), dtype=torch.bfloat16, device="cuda")
    x[..., :C] = torch.randn((B, n, C), device="cuda", generator=g).to(torch.bfloat16)
    y = torch.full((B, C, ld), 5.0, dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_transpose_bnc(p(x), padc(C), p(y), ld, B, n, C, S()))
    torch.cuda.synchronize()
    assert torch.equal(y[..., :n], x[..., :C].transpose(1, 2)) and (y[..., n:] == 0).all()


@pytest.mark.parametrize("N,Cc,H,W,ks,stride,pad,ldy", [(3, 4, 32, 32, 3, 2, 1, 48), (2, 3, 17, 23, 3, 2, 1, 32),
                                                          (2, 7, 16, 16, 3, 1, 1, 64), (1, 4, 8, 8, 1, 1, 0, 8)])
def test_im2col_is_unfold(N, Cc, H, W, ks, stride, pad, ldy):
    """b2u_im2col == torch.nn.functional.unfold (lane = c*ks*ks + ky*ks + kx, zeros outside the image and in the pad lanes):
    a pure gather, bit-exact; with the weight [Cout][Cin][kh][kw] read as rows of Cin*kh*kw the 1x1 product over these lanes
    is the convolution itself (the im2col stem of UNetB200)."""
    L, _lib = lib()
    x = rnd(N, Cc, H, W, seed=3)
    xn = nhwc(x)
    Ho, Wo = (H + 2 * pad - ks) // stride + 1, (W + 2 * pad - ks) // stride + 1
    y = torch.full((N, Ho, Wo, ldy), 7.0, dtype=torch.bfloat16, device="cuda")
    _lib.check(L.b2u_im2col(xn.data_ptr(), xn.shape[-1], Cc, N, H, W, ks, stride, pad, y.data_ptr(), ldy, None), "b2u_im2col")
    ref = F.unfold(x, ks, padding=pad, stride=stride).view(N, Cc * ks * ks, Ho, Wo).permute(0, 2, 3, 1)
    assert torch.equal(y[..., :Cc * ks * ks].float(), ref)
    assert (y[..., Cc * ks * ks:] == 0).all()
    w = rnd(5, Cc, ks, ks, seed=4)
    conv = F.conv2d(x, w, stride=stride, padding=pad).permute(0, 2, 3, 1)
    assert rel(y[..., :Cc * ks * ks].float() @ w.view(5, -1).t(), conv) < 1e-5
