"""Model-level GPU parity: the libb2u.so launch plan vs the oracle (same weights, same inputs), through the public
network API (which calls the C-ABI for every kernel).

Stated tolerances (bf16 storage, fp32 accumulation; errors are max|a-b| / max|b| per tensor):
  * logits vs the fp32 oracle            <= 3e-2   (stock torch bf16 autocast measures 2.0-2.4e-2 on the same inputs);
    for xresnet50 <= max(3e-2, 1.25 x the autocast error measured in the same test) - autocast reads 5.6-5.8e-2 there
    and this pipeline 5.3-6.2e-2 (tools/parity_probe.py xresnet50 4 8 64 2)
  * loss vs the fp32 oracle              <= 5e-3
  * logits vs the bf16-storage emulation <= 2e-2 and loss <= 2e-4 (5e-4 for xresnet50; same rounding points: only accumulation order and
    rounding-boundary flips differ)
  * argmax masks: every disagreement with the fp32 oracle lies where the oracle's top-2 margin is below twice the
    measured logit error; >= 99.9 % agreement on pixels with a larger margin (north_star's 99.9 % bar)
  * parameter gradients, the check that pins the wiring: against the TEACHER-FORCED bf16 emulation
    (oracle/bf16_emulation.py `taps=`: the emulation's forward values are pinned to the plan's stored activations, its
    backward rounds where the plan stores bf16) every tensor agrees within GRAD_TOL in the relative L2 norm (measured:
    1.0-2.1e-2; GRAD_TOL_DEEP for xresnet50: 3.0e-2), with cosine >= GRAD_COS and no element off by more than GRAD_TOL_MAX of the tensor maximum (measured
    1.2-6.7e-2: the max-norm follows single rounding flips, whose realisation changes with any change of summation
    order in the forward pass); tensors of fewer than 16 elements (SelfAttention gamma: one cancelling sum) pass up to
    4 x their own measured sensitivity to sub-ulp perturbations of the stored gradients.  The same checker is then run
    on copies with one weight gradient zeroed, sign-flipped and scaled by 1.05 and must flag exactly that tensor (the
    suite is known to be able to fail).  Under teacher forcing every stored forward activation must also
    equal what the emulation computes from the plan's previous activations within 2 bf16 ulp of the tensor maximum
    (a per-layer forward wiring check), and the logits within 1e-4.
  * parameter gradients vs the fp32 oracle: err(ours) <= 1.6 * err(torch bf16 autocast vs fp32) + 2e-2 on every tensor
    that stock autocast itself resolves to better than 50 %; the free-running comparison has no power beyond that
    (the network is chaotic at random init: tests/test_cpu.py::test_teacher_forced_emulation), which is why the
    teacher-forced check above exists.  Gradients are bit-identical on a re-run.
"""
import copy
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


from parity_util import gradient_mismatches, plan_taps, rel

GRAD_TOL, GRAD_COS = 3e-2, 0.999      # plan vs teacher-forced emulation, every parameter tensor: relative L2 error, cosine
GRAD_TOL_DEEP = 4e-2                  # xresnet50 / 101 (50+ stored tensors per path; measured 2.7-3.0e-2)
GRAD_TOL_MAX = 1e-1                   # ... and the largest single-element error relative to the tensor maximum
ACT_TOL = 2 * 2.0 ** -8               # stored activation vs the emulation's value from the plan's previous activations


def teacher_forced_check(oracle, net, x, yl, w, logits):
    """Gradients of the teacher-forced emulation vs the plan's, per-layer forward consistency, mutation self-test."""
    from oracle.bf16_emulation import emulated_forward
    from oracle.unet_oracle import weighted_ce
    o_tf = copy.deepcopy(oracle)
    o_tf.zero_grad()
    taps, free, mism = plan_taps(net), {}, {}
    l_tf = emulated_forward(o_tf, x, True, taps=taps, record=free, mismatch=mism)
    weighted_ce(l_tf, yl, w).backward()
    assert rel(logits, l_tf) <= 1e-4, rel(logits, l_tf)
    assert len(free) >= 40
    # (`layers.8.0.out` is not materialised when the final PixelShuffle is fused into its convolution: it is checked
    # through `layers.10.cat`'s consumers instead)
    assert len(mism) >= len(free) - 1
    off = {k: e for k, e in mism.items() if e > ACT_TOL}
    assert not off, sorted(off.items(), key=lambda kv: -kv[1])[:5]
    ref = {n: p.grad for n, p in o_tf.named_parameters()}
    grads = net.named_grads()
    # tensors that are ONE cancelling sum: how far the reference itself moves under a 2^-9 relative perturbation in front
    # of every backward rounding (forward values stay pinned by the taps)
    tiny = [n for n in ref if ref[n].numel() < 16]
    floors = {}
    if tiny:
        o_n = copy.deepcopy(oracle)
        o_n.zero_grad()
        torch.manual_seed(1234)
        weighted_ce(emulated_forward(o_n, x, True, taps=taps, noise=2.0 ** -9), yl, w).backward()
        g_n = {n: p.grad for n, p in o_n.named_parameters()}
        floors = {n: rel(g_n[n], ref[n]) for n in tiny}
    tol = GRAD_TOL_DEEP if oracle.arch in ("xresnet50", "xresnet101") else GRAD_TOL
    check = lambda g: gradient_mismatches(g, ref, tol, GRAD_COS, GRAD_TOL_MAX, floors)
    bad = check(grads)
    assert not bad, (sorted(bad, key=lambda b: -b[1])[:10], floors)
    # the checker can fail: one zeroed / sign-flipped / 5 %-scaled weight gradient is flagged, and only that tensor
    names = [n for n in ref if n.endswith("convpath.1.0.weight") and n.startswith("layers.0.7.")]
    victim = names[-1]
    for mutate in (torch.zeros_like, lambda g: -g, lambda g: 1.05 * g):
        broken = dict(grads)
        broken[victim] = mutate(grads[victim])
        assert [b[0] for b in check(broken)] == [victim]
    from parity_util import rel_l2
    worst = max(rel(grads[n], ref[n]) for n in ref if n not in floors)
    worst2 = max(rel_l2(grads[n], ref[n]) for n in ref if n not in floors)
    if os.path.isdir("gpurun_out"):      # calibration record of the evidence runs (not part of the assertion)
        with open("gpurun_out/tf_parity.txt", "a") as f:
            f.write(f"{oracle.arch} {tuple(x.shape)}: worst grad err vs teacher-forced emulation L2 {worst2:.3e} max-norm "
                    f"{worst:.3e}, worst activation mismatch {max(mism.values()):.3e}, floors {floors}\n")
    return worst


def _setup(arch, n_in, n_out, size, batch, data):
    from oracle.unet_oracle import make_oracle
    from unet_b200.network import UNetB200
    from unet_b200.synth import aerial_like_tiles, uniform_tiles
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    oracle = make_oracle(arch, n_in, n_out, seed=0).cuda()
    net = UNetB200(arch, n_in, n_out, (size, size), batch, training=True)
    net.load_state_dict(oracle.state_dict())
    x_u8, y = (uniform_tiles if data == "uniform" else aerial_like_tiles)(batch, n_in, size, size, n_out)
    return oracle, net, x_u8.cuda(), y.cuda()


CASES = [("xresnet34", 4, 2, 256, 2, "uniform"), ("xresnet34", 4, 2, 128, 4, "aerial"),
         ("xresnet18", 3, 2, 128, 8, "aerial"), ("xresnet34", 4, 5, 64, 4, "aerial"),
         ("xresnet50", 4, 8, 64, 2, "aerial"),   # bottleneck blocks, 2048-wide encoder, 8 classes (BASELINE configs[3])
         # odd extents: 72 -> 36,18,9,5,3: two AvgPool(ceil_mode) idpaths on odd inputs and two decoder crops (6 vs 5,
         # 10 vs 9 == F.interpolate nearest); 75 adds an odd tile itself (stem on odd planes, final ResizeToOrig crop)
         ("xresnet18", 4, 2, 72, 4, "aerial"), ("xresnet34", 4, 3, 75, 2, "aerial"),
         ("xresnet34", 4, 2, 400, 1, "aerial")]  # the reference's default patch_size (params_and_main.py:36): 25 -> 13 -> 26 vs 25


@pytest.mark.parametrize("arch,n_in,n_out,size,batch,data", CASES)
def test_train_step_parity(arch, n_in, n_out, size, batch, data):
    from oracle.bf16_emulation import emulated_forward
    from oracle.unet_oracle import weighted_ce
    oracle, net, x_u8, y = _setup(arch, n_in, n_out, size, batch, data)
    oracle.train()
    x = x_u8.float() / 255.0
    yl = y.long()
    w = torch.full((n_out,), 1.0 / n_out, device="cuda")
    o_auto, o_emu = copy.deepcopy(oracle), copy.deepcopy(oracle)
    logits_ref = oracle(x)
    loss_ref = weighted_ce(logits_ref, yl, w)
    loss_ref.backward()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        l_auto = o_auto(x)
    weighted_ce(l_auto.float(), yl, w).backward()
    l_emu = emulated_forward(o_emu, x, True)
    loss_emu = weighted_ce(l_emu, yl, w)

    net.set_input(x_u8)
    net.set_labels(y)
    net.forward()
    loss = net.loss_and_grad()
    net.backward()
    torch.cuda.synchronize()
    logits = net.logits_nchw()

    e_logits = rel(logits, logits_ref)
    # xresnet50 (50+ bf16 rounding points per path, 2048-wide sums): stock autocast itself measures 5.6-5.8e-2 there, so
    # the bound follows torch's own bf16 error when that exceeds the flat 3e-2
    e_auto = rel(l_auto.float(), logits_ref)
    assert e_logits <= max(3e-2, 1.25 * e_auto), (e_logits, e_auto)
    assert abs(loss.item() - loss_ref.item()) / abs(loss_ref.item()) <= 5e-3
    assert rel(logits, l_emu) <= (3e-2 if arch == "xresnet50" else 2e-2)
    # (xresnet50 at batch 2 / 64 px normalises over 8 values in its last stage: the fp32 summation order of the batch
    # statistics alone moves the loss by 1-3e-4 there - measured with two orders of the same sums)
    assert abs(loss.item() - loss_emu.item()) / abs(loss_emu.item()) <= (5e-4 if arch == "xresnet50" else 2e-4)
    # argmax: disagreements only inside the error band
    top2 = logits_ref.topk(2, dim=1).values
    margin = top2[:, 0] - top2[:, 1]
    band = 2 * e_logits * logits_ref.abs().max()
    differ = logits.argmax(1) != logits_ref.argmax(1)
    assert not (differ & (margin > band)).any()
    clear = margin > band
    assert (~differ)[clear].float().mean().item() >= 0.999
    # running statistics follow torch's update rule (momentum 0.1, unbiased variance)
    sd = oracle.state_dict()
    for k, b in net.buffers.items():
        # deep stages average over few samples (e.g. 4x4x4 at 1/32 resolution).  The xresnet50 case has 8-32 samples per
        # channel behind 40+ bf16 layers: its batch variances move by tens of percent between ANY two bf16 pipelines
        # (the running update scales that by the momentum 0.1), so only gross errors are caught there
        shallow = k.startswith(("layers.0.0", "layers.0.1", "layers.0.2", "layers.0.4", "layers.0.5", "layers.6", "layers.7"))
        deep = arch == "xresnet50" and not shallow
        assert rel(b, sd[k]) <= (0.3 if deep else 5e-2), k
    # gradients: (1) against the teacher-forced emulation - tight on every tensor, with a mutation self-test
    teacher_forced_check(oracle, net, x, yl, w, logits)
    # (2) against the fp32 oracle, calibrated with torch's own bf16 autocast, where autocast itself resolves the tensor
    grads, pa = net.named_grads(), dict(o_auto.named_parameters())
    bad = []
    for name, p in oracle.named_parameters():
        eo, ea = rel(grads[name], p.grad), rel(pa[name].grad, p.grad)
        if ea <= 0.5 and eo > 1.6 * ea + 2e-2:
            bad.append((name, eo, ea))
    assert not bad, bad[:10]
    # determinism: a second forward/backward over the same inputs reproduces every gradient bit for bit (fixed-order
    # reductions, no float atomics) - a race in a grid barrier or a split-K reduce would show up here
    g1 = net.grads.clone()
    net.forward()
    net.loss_and_grad()
    net.backward()
    torch.cuda.synchronize()
    assert torch.equal(g1, net.grads)


def test_self_attention_parity():
    """self_attention=True (the reference's default, params_and_main.py:83): fastai SelfAttention on UnetBlock #1 with
    spectral-normed query / key / value convolutions - logits, loss, every gradient (incl. gamma and the weight_orig
    tensors behind the spectral norm), the power-iteration vectors, and the eval-mode forward against the oracle."""
    from oracle.unet_oracle import make_oracle, weighted_ce
    from unet_b200.network import UNetB200
    from unet_b200.synth import aerial_like_tiles
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    arch, n_in, n_out, size, batch = "xresnet18", 4, 2, 128, 4
    oracle = make_oracle(arch, n_in, n_out, seed=0, self_attention=True).cuda().train()
    o_init = copy.deepcopy(oracle)        # (a training-mode forward advances the power-iteration vectors in place)
    net = UNetB200(arch, n_in, n_out, (size, size), batch, training=True, self_attention=True)
    sd0 = copy.deepcopy(oracle.state_dict())
    net.load_state_dict(sd0)
    x_u8, y = aerial_like_tiles(batch, n_in, size, size, n_out)
    x_u8, y = x_u8.cuda(), y.cuda()
    x, yl = x_u8.float() / 255.0, y.long()
    w = torch.full((n_out,), 1.0 / n_out, device="cuda")
    o_auto = copy.deepcopy(oracle)
    logits_ref = oracle(x)
    loss_ref = weighted_ce(logits_ref, yl, w)
    loss_ref.backward()
    with torch.autocast("cuda", dtype=torch.bfloat16):
        l_auto = o_auto(x)
    weighted_ce(l_auto.float(), yl, w).backward()
    net.set_input(x_u8)
    net.set_labels(y)
    net.forward()
    loss = net.loss_and_grad()
    net.backward()
    torch.cuda.synchronize()
    logits = net.logits_nchw()
    e_logits, e_auto = rel(logits, logits_ref), rel(l_auto.float(), logits_ref)
    assert e_logits <= max(3e-2, 1.25 * e_auto), (e_logits, e_auto)
    assert abs(loss.item() - loss_ref.item()) / abs(loss_ref.item()) <= 5e-3
    sd = oracle.state_dict()
    for k, b in net.buffers.items():
        if k.endswith(("weight_u", "weight_v")):          # one power iteration in fp32 on both sides
            assert rel(b, sd[k]) <= 1e-4, k
    grads, pa = net.named_grads(), dict(o_auto.named_parameters())
    bad = []
    for name, p in oracle.named_parameters():
        eo, ea = rel(grads[name], p.grad), rel(pa[name].grad, p.grad)
        # (tensors that stock autocast itself misses by more than 10 % - the scalar gamma, one cancelling sum, reads 17 %
        # there - say nothing either way in a free-running comparison)
        if ea <= 0.1 and eo > 1.6 * ea + 2e-2:
            bad.append((name, eo, ea))
    assert not bad, bad[:10]
    sa_names = [n for n in grads if ".conv2.2." in n]
    assert len(sa_names) == 4 and all(grads[n].abs().max() > 0 for n in sa_names)
    # the wiring of the block (gamma, the weight_orig tensors behind sigma, the order in which the four consumers of
    # conv2's output accumulate their gradients) against the teacher-forced emulation of the same graph
    teacher_forced_check(o_init, net, x, yl, w, logits)
    # eval mode: sigma from the stored u / v, no power iteration
    oracle.eval()
    ev = UNetB200(arch, n_in, n_out, (size, size), batch, training=False, self_attention=True)
    ev.load_state_dict(oracle.state_dict())
    ev.set_input(x_u8)
    ev.forward()
    torch.cuda.synchronize()
    with torch.no_grad():
        ref_eval = oracle(x)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            auto_eval = oracle(x).float()
    e_ev, e_ev_auto = rel(ev.logits_nchw(), ref_eval), rel(auto_eval, ref_eval)
    # the same network without the attention block, same weights otherwise: the block must not add error of its own
    o_plain = make_oracle(arch, n_in, n_out, seed=0).cuda().eval()
    o_plain.load_state_dict({k: v for k, v in oracle.state_dict().items() if ".conv2.2." not in k})
    ev_plain = UNetB200(arch, n_in, n_out, (size, size), batch, training=False)
    ev_plain.load_state_dict(o_plain.state_dict())
    ev_plain.set_input(x_u8)
    ev_plain.forward()
    torch.cuda.synchronize()
    with torch.no_grad():
        e_plain = rel(ev_plain.logits_nchw(), o_plain(x))
    assert e_ev <= max(3e-2, 1.25 * e_ev_auto, 1.5 * e_plain), (e_ev, e_ev_auto, e_plain)
    assert torch.equal(ev.buffers["layers.5.conv2.2.query.0.weight_u"], oracle.state_dict()["layers.5.conv2.2.query.0.weight_u"])


def test_eval_forward_and_tile_prediction():
    from oracle.unet_oracle import make_oracle
    from unet_b200.network import UNetB200
    from unet_b200.predict_engine import TiledPredictor
    from unet_b200.synth import aerial_like_tiles
    torch.backends.cudnn.allow_tf32 = False
    oracle = make_oracle("xresnet34", 4, 2).cuda().eval()
    net = UNetB200("xresnet34", 4, 2, (256, 256), 2, training=False)
    net.load_state_dict(oracle.state_dict())
    x_u8, _ = aerial_like_tiles(2, 4, 256, 256, 2)
    x_u8 = x_u8.cuda()
    with torch.no_grad():
        ref = oracle(x_u8.float() / 255.0)
    probs, amax = TiledPredictor(net).predict_tiles(x_u8)
    got = net.logits_nchw()
    torch.cuda.synchronize()
    e = rel(got, ref)
    assert e <= 3e-2, e
    # the softmax kernel itself (fp32 in, fp32 out) against torch on the SAME logits; with random-init weights the
    # logits reach +-90, where a 2.5 % logit error moves saturated probabilities arbitrarily, so probabilities are not
    # compared with the oracle's directly
    assert rel(probs, got.softmax(1)) <= 1e-5
    assert torch.equal(amax.long(), got.argmax(1))
    top2 = ref.topk(2, dim=1).values
    margin = top2[:, 0] - top2[:, 1]
    differ = amax.long() != ref.argmax(1)
    assert not (differ & (margin > 2 * e * ref.abs().max())).any()


def test_predict_raster_matches_reference_merge():
    """Tiled predict-and-stitch of a small raster: GPU mask vs the numpy merge (predict.py:284-337 restated) fed with
    the oracle's per-tile softmax probabilities; also checks that a 2-way column sharding reproduces the 1-GPU mask
    bit-exactly (owner-computes strips).  At overlap 0.75 a tile overlaps three neighbours per axis: batches then need
    more than 2 x 2 colour classes."""
    import numpy as np
    from oracle.stitch import merge_pixel_windows
    from oracle.unet_oracle import make_oracle
    from unet_b200.network import UNetB200
    from unet_b200.predict_engine import TiledPredictor
    from unet_b200.tiling import colour_classes, compute_windows
    torch.backends.cudnn.allow_tf32 = False
    P, H, W = 64, 200, 264
    oracle = make_oracle("xresnet18", 4, 2).cuda().eval()
    net = UNetB200("xresnet18", 4, 2, (P, P), 8, training=False)
    net.load_state_dict(oracle.state_dict())
    g = torch.Generator().manual_seed(3)
    low = torch.rand((4, 8, 9), generator=g)
    raster = (torch.nn.functional.interpolate(low[None], size=(H, W), mode="bilinear")[0] * 255).round().to(torch.uint8)
    raster = raster.cuda().contiguous()
    pred = TiledPredictor(net)
    for ov in (0.125, 0.75):
        mask, xb, xe = pred.predict_raster(raster, ov)
        torch.cuda.synchronize()
        wins = compute_windows(H, W, P, ov)
        if ov > 0.5:
            assert max(len(colour_classes(wins[b:b + 8])) for b in range(0, len(wins), 8)) > 4
        probs = []
        with torch.no_grad():
            for (x, y, w, h) in wins:
                t = raster[:, y:y + h, x:x + w][None].float() / 255.0
                probs.append(oracle(t).softmax(1)[0].cpu().numpy())
        ref = merge_pixel_windows(probs, wins, H, W)
        agree = (mask.cpu().numpy() == ref).mean()
        assert agree >= 0.995, (ov, agree)  # random-init logits are near-ties almost everywhere; see test docstring above
        # sharded == single GPU, bit-exact
        parts = []
        for r in range(2):
            m, b, e = pred.predict_raster(raster, ov, rank=r, world=2)
            parts.append(m)
        torch.cuda.synchronize()
        assert torch.equal(torch.cat(parts, dim=1), mask)
        # 2 x 2 ownership grid (what 8 GPUs use as 4 x 2): every cell equals the same window of the 1-GPU mask
        for r in range(4):
            m, (xb, xe, yb, ye) = pred.predict_raster(raster, ov, rank=r, world=4, grid=(2, 2))
            assert torch.equal(m, mask[yb:ye, xb:xe])


def test_against_committed_golden_fixture():
    """tests/golden/model_xresnet18_32.npz (generated by tests/golden/make_golden.py from the oracle): logits of the
    train-mode and eval-mode forward for fixed inputs; the CUDA plan must reproduce them within the bf16 tolerance."""
    import numpy as np
    from oracle.unet_oracle import make_oracle
    from unet_b200.network import UNetB200
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "model_xresnet18_32.npz"))
    oracle = make_oracle("xresnet18", 3, 2, seed=0)
    x_u8 = torch.from_numpy(g["x_u8"]).cuda()
    for training, key in ((True, "logits_train"), (False, "logits_eval")):
        net = UNetB200("xresnet18", 3, 2, (32, 32), 2, training=training)
        net.load_state_dict(oracle.state_dict())
        net.set_input(x_u8)
        net.forward()
        torch.cuda.synchronize()
        e = rel(net.logits_nchw().cpu(), torch.from_numpy(g[key]))
        assert e <= 3e-2, (key, e)
