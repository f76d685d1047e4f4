"""The strict-precision training plan on the B200: its new kernels against torch on seeded inputs, its train-mode forward against
the fp32 oracle (logits, every feature, the Lovasz loss, ReLU masks), its gradients against plain fp32 autograd, graph replay and
determinism, `UNet.train_precision`, the weight-overflow rebuild, the config-5 plan and `rs train` with RSB_TRAIN_PRECISION=strict."""

import argparse

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import losses_oracle, unet_oracle
from robosat_b200 import _lib, synth
from robosat_b200.train_engine import UNetTrainEngine

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = a.double(), b.double()
    return ((a - b).pow(2).sum().sqrt() / b.pow(2).sum().sqrt().clamp_min(1e-30)).item()


def _split(v32):
    hi = v32.half()
    return torch.stack([hi, (v32 - hi.float()).half()])


def _pair(t):
    return t[0].float() + t[1].float()


def _engine(C, B, S, device, precision="strict", loss_scale=1024.0):
    sd0 = {k[7:]: v.clone() for k, v in synth.make_state_dict(C, seed=0).items()}
    x = synth.normalize_tiles(synth.make_tiles_u8(B, S, seed=1))
    params = {k: v.clone().to(device) for k, v in sd0.items()}
    return sd0, x, params, UNetTrainEngine(params, C, B, S, S, device=device, loss_scale=loss_scale, precision=precision)


def _nchw(eng, t, shape):
    """fp32 NCHW value of an engine activation (hi + lo for a two-plane buffer), dec4's W padding removed"""
    n, h, w, c = shape
    v = _pair(t) if eng.strict else t.float()
    v = v.reshape(n, h, w, c)
    if w == eng.W + 4:
        v = v[:, :, 1:eng.W + 1]
    return v.permute(0, 3, 1, 2).cpu()


# ------------------------------------------------------------------------------------------------ kernels
def test_pack_weights_split_bits_and_overflow_counter(cuda_device):
    lib, st, d = _lib.load(), _lib.current_stream_ptr(), cuda_device
    g = torch.Generator().manual_seed(0)
    src = torch.randn(4096, generator=g) * 0.05
    src[17] = 1e6  # past any exponent that fits the others
    n = 2048
    map4 = torch.randint(-1, 4096, (n, 4), generator=g, dtype=torch.int32)
    map1 = torch.randint(-1, 4096, (n,), generator=g, dtype=torch.int32)
    scale = 2.0 ** 13
    for single, m in ((False, map4), (True, map1)):
        mm = m.long().reshape(n, -1)
        v = torch.zeros(n)
        for j in range(mm.shape[1]):
            v = v + torch.where(mm[:, j] >= 0, src[mm[:, j].clamp_min(0)], torch.zeros(()))
        ref = _split(v * scale)
        bad = ~((v * scale).abs() < 65520)
        srcd, md = src.to(d), m.to(d)
        dst = torch.zeros((2, n), dtype=torch.float16, device=d)
        cnt = torch.full((1,), 5, dtype=torch.int32, device=d)  # the counter accumulates
        fn = lib.rsb_pack_weights1_split if single else lib.rsb_pack_weights_split
        _lib.check(fn(srcd.data_ptr(), md.data_ptr(), dst.data_ptr(), n, n, scale, cnt.data_ptr(), st), "pack_split")
        torch.cuda.synchronize()
        got = dst.cpu()
        assert int(bad.sum()) >= 1
        assert int(cnt.item()) == 5 + int(bad.sum())
        ok = ~bad
        assert torch.equal(got[0][ok].view(torch.int16), ref[0][ok].view(torch.int16)), single
        assert torch.equal(got[1][ok].view(torch.int16), ref[1][ok].view(torch.int16)), single
        assert torch.isinf(got[0][bad]).all()
    # arguments are validated
    assert lib.rsb_pack_weights1_split(srcd.data_ptr(), md.data_ptr(), dst.data_ptr(), n, n - 1, scale, cnt.data_ptr(), st) == -1
    assert lib.rsb_pack_weights_split(srcd.data_ptr(), md.data_ptr(), dst.data_ptr(), n - 1, n, scale, cnt.data_ptr(), st) == -1


def test_bn_stats_and_apply_split(cuda_device):
    lib, st, d = _lib.load(), _lib.current_stream_ptr(), cuda_device
    g = torch.Generator().manual_seed(1)
    for (M, C, res) in [(2 * 16 * 16, 64, False), (3 * 8 * 8, 2048, True), (4 * 96 * 96, 128, True), (5 * 7 * 9, 256, False)]:
        v = torch.randn((M, C), generator=g) * 1.5 + 0.3
        z = _split(v)
        zv = _pair(z).double()
        gamma, beta = torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g) * 0.1
        rm, rv = torch.randn(C, generator=g) * 0.1, torch.rand(C, generator=g) + 0.5
        zd, gd, bd, rmd, rvd = z.to(d), gamma.to(d), beta.to(d), rm.to(d), rv.to(d)
        nb = torch.zeros((), dtype=torch.int64, device=d)
        sums = torch.zeros(20 * C, dtype=torch.float64, device=d)
        mean, invstd, scale, shift = (torch.zeros(C, device=d) for _ in range(4))
        _lib.check(lib.rsb_bn_stats_finalize_split(zd.data_ptr(), M * C, sums.data_ptr(), gd.data_ptr(), bd.data_ptr(), rmd.data_ptr(), rvd.data_ptr(),
                                                   nb.data_ptr(), mean.data_ptr(), invstd.data_ptr(), scale.data_ptr(), shift.data_ptr(), M, C,
                                                   1e-5, 0.1, None, st), "stats_split")
        torch.cuda.synchronize()
        slots = sums[:16 * C].reshape(8, 2, C).sum(0).cpu()
        s0, s1 = zv.sum(0), (zv * zv).sum(0)
        assert ((slots[0] - s0).abs() <= 1e-12 * zv.abs().sum(0)).all()
        assert ((slots[1] - s1).abs() <= 1e-12 * s1).all()
        mu = s0 / M
        var = s1 / M - mu * mu
        istd = 1.0 / torch.sqrt(var + 1e-5)
        assert torch.allclose(mean.cpu().double(), mu, rtol=1e-6, atol=1e-7) and torch.allclose(invstd.cpu().double(), istd, rtol=1e-6)
        assert torch.allclose(scale.cpu(), gamma * istd.float(), rtol=1e-6) and torch.allclose(shift.cpu(), beta - mu.float() * gamma * istd.float(),
                                                                                               rtol=1e-5, atol=1e-6)
        assert torch.allclose(rmd.cpu().double(), 0.9 * rm.double() + 0.1 * mu, rtol=1e-6, atol=1e-7)
        assert torch.allclose(rvd.cpu().double(), 0.9 * rv.double() + 0.1 * var * M / (M - 1), rtol=1e-6)
        assert int(nb.item()) == 1
        # chained variant: same outputs, slots left zeroed
        rm2, rv2 = rm.to(d), rv.to(d)
        nb2 = torch.zeros((), dtype=torch.int64, device=d)
        sums2 = torch.zeros_like(sums)
        outs2 = [torch.zeros(C, device=d) for _ in range(4)]
        _lib.check(lib.rsb_bn_stats_finalize_split_chained(zd.data_ptr(), M * C, sums2.data_ptr(), gd.data_ptr(), bd.data_ptr(), rm2.data_ptr(),
                                                           rv2.data_ptr(), nb2.data_ptr(), *[o.data_ptr() for o in outs2], M, C, 1e-5, 0.1, None, st), "chained")
        torch.cuda.synchronize()
        for got, want in zip(outs2 + [rm2, rv2], [mean, invstd, scale, shift, rmd, rvd]):
            assert torch.allclose(got, want, rtol=1e-6, atol=1e-7)
        assert not sums2[:16 * C + 2].any()

        # apply: y = relu(z*scale + shift (+ r)) in fp32, split. Reference: the same fp32 operations (fma through fp64, exact
        # product), split the same way; compared on hi + lo within one fp32 ulp of the value (plus what an fp32 ulp of y moves lo by)
        r = _split(torch.randn((M, C), generator=g)) if res else None
        sc, sh = scale.cpu(), shift.cpu()
        o = (_pair(z).double() * sc.double() + sh.double()).float()
        if res:
            o = o + _pair(r)
        want = _pair(_split(torch.relu(o)))
        y = torch.zeros((2, M, C), dtype=torch.float16, device=d)
        rd = r.to(d) if res else None
        _lib.check(lib.rsb_bn_apply_split(zd.data_ptr(), M * C, scale.data_ptr(), shift.data_ptr(), rd.data_ptr() if res else None, M * C if res else 0,
                                          y.data_ptr(), M * C, M, C, 1, st), "apply_split")
        torch.cuda.synchronize()
        got = _pair(y.cpu())
        ulp = torch.where(want.abs() > 0, want.abs() * 2.0 ** -23, torch.full_like(want, 2.0 ** -149))
        diff = (got - want).abs()
        print("bn_apply_split M=%d C=%d: %d of %d differ, worst %.2f ulp" % (M, C, int((diff > 0).sum()), diff.numel(), float((diff / ulp).max())))
        assert (diff <= 4 * ulp).all() and float((diff > ulp).float().mean()) < 1e-3
        assert torch.equal(got > 0, want > 0)


def test_maxpool_backward_split_routes_by_hi_plus_lo(cuda_device):
    lib, st, d = _lib.load(), _lib.current_stream_ptr(), cuda_device
    g = torch.Generator().manual_seed(2)
    for (N, H, W, C, k, s, p) in [(2, 16, 16, 64, 3, 2, 1), (2, 4, 4, 128, 2, 2, 0), (3, 10, 14, 8, 3, 2, 1)]:
        # coarse values (many hi ties inside a window) + residues below half an fp16 ulp (the lo planes decide), and exact ties
        base = torch.relu(torch.randint(-2, 3, (N, H, W, C), generator=g).float())
        v = base + torch.rand((N, H, W, C), generator=g) * 2.0 ** -13 * (base > 0)
        x = _split(v)
        assert torch.equal(x[0].float(), base)  # every hi is the coarse value: only lo tells the windows' elements apart
        vn = _pair(x).permute(0, 3, 1, 2).contiguous().requires_grad_(True)
        yy = F.max_pool2d(vn, k, s, p)
        dy = torch.randn(yy.shape, generator=g).half()
        yy.backward(dy.float())
        want = vn.grad.permute(0, 2, 3, 1).half()
        xd, dyd = x.to(d), dy.permute(0, 2, 3, 1).contiguous().to(d)
        scratch = torch.zeros(dyd.numel(), dtype=torch.uint8, device=d)
        dx = torch.zeros((N, H, W, C), dtype=torch.float16, device=d)
        _lib.check(lib.rsb_maxpool_backward_split(xd.data_ptr(), x[0].numel(), dyd.data_ptr(), dx.data_ptr(), scratch.data_ptr(), N, H, W, C, k, s, p, st),
                   "maxpool_bwd_split")
        hi_only = torch.zeros_like(dx)
        _lib.check(lib.rsb_maxpool_backward(xd.data_ptr(), dyd.data_ptr(), hi_only.data_ptr(), scratch.data_ptr(), N, H, W, C, k, s, p, st), "maxpool_bwd")
        torch.cuda.synchronize()
        assert torch.allclose(dx.cpu().float(), want.float(), atol=2e-3, rtol=2e-3)
        assert not torch.equal(hi_only.cpu(), dx.cpu())  # the single-plane arg-max routes differently: the test is not vacuous


def test_final_forward_split(cuda_device):
    lib, st, d = _lib.load(), _lib.current_stream_ptr(), cuda_device
    g = torch.Generator().manual_seed(4)
    for C, N, HW in [(2, 2, 64 * 64), (6, 1, 32 * 48)]:
        y5 = _split(torch.relu(torch.randn((N * HW, 32), generator=g)))
        w, b = torch.randn((C, 32), generator=g) * 0.2, torch.randn(C, generator=g)
        logits = torch.zeros((N, C, HW), device=d)
        yd, wd, bd = y5.to(d), w.to(d), b.to(d)
        ovf = torch.zeros(1, dtype=torch.int32, device=d)
        _lib.check(lib.rsb_final_forward_split(yd.data_ptr(), N * HW * 32, wd.data_ptr(), bd.data_ptr(), ovf.data_ptr(), logits.data_ptr(), N, HW, C, st),
                   "final_split")
        torch.cuda.synchronize()
        ref = (_pair(y5).double().reshape(N, HW, 32) @ w.double().t() + b.double()).permute(0, 2, 1)
        assert _rel(logits.cpu(), ref) < 1e-6
        ovf.fill_(1)  # the pack counted weights past the plan's exponents: the logits are poisoned
        _lib.check(lib.rsb_final_forward_split(yd.data_ptr(), N * HW * 32, wd.data_ptr(), bd.data_ptr(), ovf.data_ptr(), logits.data_ptr(), N, HW, C, st),
                   "final_split")
        torch.cuda.synchronize()
        assert torch.isnan(logits).all()


# ------------------------------------------------------------------------------------------------ the strict plan vs the oracle
def _relu_outputs_of_oracle(monkeypatch, sd, x):
    """the oracle's train-mode forward, recording every F.relu output in call order (stem, per block relu1 / relu2 / out, center,
    dec0..dec4, dec5: the order of UNetTrainEngine.relu_outs)"""
    seen = []
    relu = F.relu

    def rec(t, *a, **k):
        out = relu(t, *a, **k)
        seen.append(out)
        return out

    monkeypatch.setattr(torch.nn.functional, "relu", rec)
    with torch.no_grad():
        logits, feats = unet_oracle.unet_forward_train(sd, x, return_features=True)
    monkeypatch.setattr(torch.nn.functional, "relu", relu)
    return logits, feats, seen


@pytest.mark.parametrize("size", [128, 512])
def test_strict_train_forward_matches_oracle(size, cuda_device, monkeypatch):
    sd0, x, params, eng = _engine(2, 2, size, cuda_device)
    logits = eng.forward(x.to(cuda_device)).float().cpu()
    sd = {k: v.clone() for k, v in sd0.items()}
    ref, feats, relus = _relu_outputs_of_oracle(monkeypatch, sd, x)
    r = _rel(logits, ref)
    worst = max((_rel(_nchw(eng, *eng.feats[n]), feats[n]), n) for n in feats)
    print("strict train-mode forward 2x%d^2: logits rel-L2 %.2e, worst feature %s" % (size, r, worst))
    assert r <= 2e-4 and worst[0] <= 2e-4
    for k in ("resnet.bn1", "resnet.layer2.0.downsample.1", "resnet.layer4.2.bn3"):
        assert _rel(params[k + ".running_mean"].cpu(), sd[k + ".running_mean"]) < 1e-4
        assert _rel(params[k + ".running_var"].cpu(), sd[k + ".running_var"]) < 1e-4
    if size != 128:
        return
    # step-0 Lovasz loss
    masks = synth.make_masks(2, size, 2, seed=3)
    from robosat_b200.losses import LovaszLoss2d

    loss = float(LovaszLoss2d().to(cuda_device)(eng.logits, masks.to(cuda_device)))
    ref_loss = float(losses_oracle.lovasz_loss(ref, masks))
    print("step-0 Lovasz loss strict %.7f oracle %.7f" % (loss, ref_loss))
    assert abs(loss - ref_loss) <= 1e-4 * abs(ref_loss)
    # ReLU masks against the oracle's, both precisions
    _, _, _, feng = _engine(2, 2, size, cuda_device, precision="fast")
    feng.forward(x.to(cuda_device))
    torch.cuda.synchronize()
    assert len(relus) == len(eng.relu_outs) == len(feng.relu_outs)
    flips = {}
    for e, name in ((eng, "strict"), (feng, "fast")):
        bad = total = 0
        for (t, shp), want in zip(e.relu_outs.values(), relus):
            got = _nchw(e, t, shp)
            assert got.shape == want.shape
            bad += int(((got > 0) != (want > 0)).sum())
            total += want.numel()
        flips[name] = bad / total
    print("ReLU mask disagreement with the oracle at 2x128^2: strict %.3e, fast %.3e (%d masks)" % (flips["strict"], flips["fast"], len(relus)))
    assert flips["strict"] * 10 <= flips["fast"]


def test_strict_backward_vs_plain_fp32_autograd(cuda_device):
    C, B, S = 2, 2, 128
    sd0, x, params, eng = _engine(C, B, S, cuda_device)
    g = torch.Generator().manual_seed(3)
    dlogits = torch.randn((B, C, S, S), generator=g) * 1e-3
    eng.forward(x.to(cuda_device))
    grads = eng.backward(dlogits.to(cuda_device))
    torch.cuda.synchronize()
    sd = {k: v.clone() for k, v in sd0.items()}
    for k, v in sd.items():
        if v.dtype == torch.float32 and "running" not in k:
            v.requires_grad_(True)
    lo = unet_oracle.unet_forward_train(sd, x)
    (lo * dlogits).sum().backward()
    rels, dots, n1, n2 = {}, 0.0, 0.0, 0.0
    for k, v in sd.items():
        if v.requires_grad and not k.startswith("resnet.fc"):
            a, b = grads[k].cpu().double(), v.grad.double()
            rels[k] = _rel(a, b)
            dots += float((a * b).sum())
            n1 += float((a * a).sum())
            n2 += float((b * b).sum())
    cosine = dots / (n1 ** 0.5 * n2 ** 0.5)
    vals = sorted(rels.values())
    worst = sorted(rels.items(), key=lambda kv: -kv[1])[:3]
    print("strict gradient vs plain fp32 autograd: median rel-L2 %.4f, 90th pct %.4f, worst %s, cosine %.6f" % (
        vals[len(vals) // 2], vals[int(0.9 * len(vals))], worst, cosine))
    assert len(rels) == 168
    assert cosine >= 0.999 and vals[len(vals) // 2] <= 3e-2 and vals[-1] <= 1e-1


def test_strict_graph_replay_and_deterministic_backward(cuda_device):
    sd0, x, params_a, eng_a = _engine(2, 2, 128, cuda_device)
    _, _, params_b, eng_b = _engine(2, 2, 128, cuda_device)
    assert eng_a.use_graph
    eng_b.use_graph = False
    g = torch.Generator().manual_seed(5)
    for step in range(4):
        xs = (x + 0.01 * step).to(cuda_device)
        dl = (torch.randn((2, 2, 128, 128), generator=g) * 1e-3).to(cuda_device)
        la = eng_a.forward(xs).clone()
        lb = eng_b.forward(xs.clone()).clone()
        ga = {k: v.clone() for k, v in eng_a.backward(dl).items()}
        gb = {k: v.clone() for k, v in eng_b.backward(dl.clone()).items()}
        torch.cuda.synchronize()
        assert torch.equal(la, lb), step
        for k in ga:
            assert torch.equal(ga[k], gb[k]), (step, k)
        if step == 3:  # a second backward over the same saved activations
            g2 = {k: v.clone() for k, v in eng_a.backward(dl).items()}
            torch.cuda.synchronize()
            for k in ga:
                assert torch.equal(ga[k], g2[k]), k
    assert any(s["graph"] is not None for s in eng_a._graphs.values())
    for k in params_a:
        if "running" in k or k.endswith("num_batches_tracked"):
            assert torch.equal(params_a[k], params_b[k]), k


def test_unet_train_precision_strict_through_dataparallel(cuda_device):
    from robosat_b200.losses import LovaszLoss2d
    from robosat_b200.optim import Adam
    from robosat_b200.unet import UNet

    sd = synth.make_state_dict(2, seed=0)
    net = torch.nn.DataParallel(UNet(2, pretrained=False), device_ids=[0]).to(cuda_device)
    net.load_state_dict(sd)
    net.module.train_precision = "strict"
    opt = Adam(net.parameters(), lr=1e-3)
    opt.mark_used([not n.startswith("module.resnet.fc.") for n, _ in net.named_parameters()])
    crit = LovaszLoss2d().to(cuda_device)
    x = synth.normalize_tiles(synth.make_tiles_u8(2, 128, seed=1)).to(cuda_device)
    masks = synth.make_masks(2, 128, 2, seed=3).to(cuda_device)
    with torch.no_grad():
        ref_logits = unet_oracle.unet_forward_train({k: v.clone() for k, v in sd.items()}, x.cpu())
    ref_loss = float(losses_oracle.lovasz_loss(ref_logits, masks.cpu()))
    net.train()
    losses = []
    for _ in range(4):
        opt.zero_grad()
        loss = crit(net(x), masks)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    print("strict lovasz losses", losses, "oracle step-0", ref_loss)
    assert [k[-1] for k in net.module._train_engines] == ["strict"]
    assert all(e.strict for e in net.module._train_engines.values())
    assert abs(losses[0] - ref_loss) <= 1e-4 * abs(ref_loss)
    assert losses[-1] < losses[0] and opt.skipped_steps() == 0
    ckpt = {"epoch": 1, "state_dict": net.state_dict(), "optimizer": opt.state_dict()}
    assert list(ckpt["state_dict"].keys()) == list(sd.keys()) and len(ckpt["optimizer"]["state"]) == 168


def test_weights_past_the_exponent_rebuild_the_plan(cuda_device):
    """A layer's weights grown past the headroom of the plan's exponent (x128 > 64x) trip the pack's overflow counter: that step's
    gradients are not finite and the guarded Adam skips it, the next forward builds a new plan, whose loss is finite and equals a
    fresh strict plan's on the same weights."""
    from robosat_b200.losses import CrossEntropyLoss2d
    from robosat_b200.optim import Adam
    from robosat_b200.unet import UNet

    sd = {k[7:]: v for k, v in synth.make_state_dict(2, seed=0).items()}
    x = synth.normalize_tiles(synth.make_tiles_u8(2, 64, seed=1)).to(cuda_device)
    masks = synth.make_masks(2, 64, 2, seed=3).to(cuda_device)
    crit = CrossEntropyLoss2d().to(cuda_device)

    def make():
        net = UNet(2, pretrained=False).to(cuda_device)
        net.load_state_dict(sd)
        net.train_precision = "strict"
        net.train()
        return net

    net = make()
    opt = Adam(net.parameters(), lr=0.0)
    losses, engines, running = [], [], []
    for step in range(3):
        if step == 1:
            with torch.no_grad():
                net.resnet.layer3[0].conv1.weight.mul_(128.0)
        running.append({k: v.clone() for k, v in net.named_buffers()})
        opt.zero_grad()
        loss = crit(net(x), masks)
        loss.backward()
        opt.step()
        losses.append(loss.item())
        engines.append(next(iter(net._train_engines.values())))
    running.append({k: v.clone() for k, v in net.named_buffers()})
    print("losses around the overflow", losses, "skipped", opt.skipped_steps())
    assert np.isfinite(losses[0]) and not np.isfinite(losses[1]) and np.isfinite(losses[2])
    assert opt.skipped_steps() == 1
    assert engines[0] is engines[1] and engines[2] is not engines[1] and not engines[2].overflowed()
    assert engines[2].exponents["resnet.layer3.0.conv1"] == engines[1].exponents["resnet.layer3.0.conv1"] - 7
    for k in running[0]:  # the tripped step left the running statistics (and batch counts) alone
        assert torch.equal(running[1][k], running[2][k]), k
    nb = "resnet.layer3.0.bn1.num_batches_tracked"
    assert int(running[3][nb]) == int(running[2][nb]) + 1 == int(running[0][nb]) + 2
    sd.update({k: v.detach().cpu() for k, v in net.state_dict().items() if "running" not in k and "num_batches" not in k})
    fresh = make()
    with torch.no_grad():
        lf = crit(fresh(x), masks).item()
    assert abs(lf - losses[2]) <= 1e-6 * abs(lf), (lf, losses[2])


def test_config5_strict_plan_batch8_1024(cuda_device):
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    sd = synth.make_state_dict(6, seed=0)
    params = {k[7:]: v.clone().to(cuda_device) for k, v in sd.items()}
    eng = UNetTrainEngine(params, 6, 8, 1024, 1024, device=cuda_device, loss_scale=4096.0, precision="strict")
    xb = synth.normalize_tiles(synth.make_tiles_u8(8, 1024, seed=2)).to(cuda_device)
    logits = eng.forward(xb)
    dl = torch.randn_like(logits) * 1e-6
    grads = eng.backward(dl)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated()
    print("cfg 5 strict plan (8 x 1024^2, 6 classes): peak %.1f GB" % (peak / 1e9))
    assert torch.isfinite(logits).all() and all(torch.isfinite(v).all() for v in grads.values())
    assert len(grads) == 168 and peak < 170e9


def test_rs_train_strict_one_epoch(tmp_path, cuda_device, monkeypatch):
    from robosat_b200.tools import train
    from test_train_tool_gpu import _write_split

    ds = tmp_path / "ds"
    _write_split(str(ds), "training", 4, 128, 1)
    _write_split(str(ds), "validation", 2, 128, 5)
    ck = tmp_path / "pth"
    (tmp_path / "model.toml").write_text("[common]\ncuda = true\nbatch_size = 2\nimage_size = 128\ncheckpoint = '%s'\n[opt]\nepochs = 1\nlr = 0.0005\nloss = 'Lovasz'\n" % ck)
    (tmp_path / "dataset.toml").write_text("[common]\ndataset = '%s'\nclasses = ['background', 'parking']\ncolors = ['denim', 'orange']\n[weights]\nvalues = [1.6248, 5.762827]\n" % ds)
    monkeypatch.setenv("RSB_GPUS", "1")
    monkeypatch.setenv("RSB_TRAIN_PRECISION", "strict")
    start = tmp_path / "start.pth"
    torch.save({"epoch": 0, "state_dict": synth.make_state_dict(2, seed=0), "optimizer": {}}, start)
    train.main(argparse.Namespace(model=str(tmp_path / "model.toml"), dataset=str(tmp_path / "dataset.toml"), checkpoint=str(start), resume=False,
                                  workers=0))
    log = open(ck / "log").read()
    assert "Epoch: 1/1" in log and "Train    loss:" in log and "Validate loss:" in log
    last = torch.load(ck / "checkpoint-00001-of-00001.pth", map_location="cpu")
    assert last["epoch"] == 1 and len(last["optimizer"]["state"]) == 168
    assert all(torch.isfinite(v).all() for k, v in last["state_dict"].items() if v.is_floating_point())
