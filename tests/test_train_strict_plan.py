"""The strict-precision training plan (UNetTrainEngine(precision="strict")) on the CPU: its op lists replayed in float64 by
`run_strict_train_ops` below match the oracle's train-mode forward at fp32 level, its descriptors are the split forms the GPU
kernels expect, and the precision is selected the way the documentation says.

`run_strict_train_ops` restates the strict-only op kinds (split weight packing, two-plane BatchNorm statistics / apply, two-plane
max-pool and its backward, the final 1x1 conv on hi + lo) with the arithmetic of their kernels, and hands every other op to
tests/emulate.py, which executes split conv descriptors with float64 contractions."""

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import emulate
from oracle import unet_oracle
from robosat_b200 import synth
from robosat_b200.train_engine import TRAIN_PRECISIONS, UNetTrainEngine, default_train_precision


def _pair_value(t):
    """fp32 value hi + lo of a two-plane buffer (exact)"""
    return t[0].float() + t[1].float()


def _store_pair(dst, v32):
    hi = v32.half()
    dst[0].copy_(hi.reshape(dst[0].shape))
    dst[1].copy_((v32 - hi.float()).half().reshape(dst[1].shape))


def _first_max_pool_bwd(v, dy, k, s, p):
    """gradient of max_pool2d routed to the first maximum of every window (row-major scan), on fp32 values: ATen's rule, and the
    one rsb_maxpool_backward_split applies to hi + lo"""
    xin = v.clone().requires_grad_(True)
    F.max_pool2d(xin, k, s, p).backward(dy)
    return xin.grad


def run_strict_train_ops(eng, ops, x=None, dlogits=None):
    """Replay a strict plan_only UNetTrainEngine op list on CPU buffers."""
    assert eng.strict and eng.plan_only
    P = eng.params
    for op in ops:
        k = op[0]
        if k == "pack_all":
            emulate.run_train_ops(eng, [op])  # the single fp16 (dgrad) layouts
            for wname, m, dst, scale, single in eng.split_pack_list:
                src = P[wname].reshape(-1)
                mm = m.long().reshape(m.shape[0], -1)
                v = torch.zeros(mm.shape[0], dtype=torch.float32)
                for j in range(mm.shape[1]):  # fp32 adds in map order, as the pack kernels do
                    v = v + torch.where(mm[:, j] >= 0, src[mm[:, j].clamp_min(0)], torch.zeros(()))
                _store_pair(dst, v * scale)
        elif k == "prepass_split":
            eng.s2d.copy_(emulate.prepass_s2d_split_cpu(x))
        elif k == "bn_stats_split":
            b = op[1]
            pf = b.prefix
            z = (b.zpair[0].double() + b.zpair[1].double()).reshape(b.M, b.C)
            mean = z.mean(0)
            var = ((z * z).sum(0) / b.M - mean * mean).clamp_min(0)
            invstd = (1.0 / torch.sqrt(var + emulate.eng_eps())).float()
            b.mean.copy_(mean.float())
            b.invstd.copy_(invstd)
            b.scale.copy_(P[pf + ".weight"] * invstd)
            b.shift.copy_(P[pf + ".bias"] - mean.float() * b.scale)
            P[pf + ".running_mean"].copy_(0.9 * P[pf + ".running_mean"] + 0.1 * mean.float())
            P[pf + ".running_var"].copy_(0.9 * P[pf + ".running_var"] + 0.1 * (var * b.M / (b.M - 1)).float())
            P[pf + ".num_batches_tracked"].add_(1)
        elif k == "bn_apply_split":
            _, b, res, y, relu = op
            o = _pair_value(b.zpair).reshape(b.M, b.C) * b.scale + b.shift
            if res is not None:
                o = o + _pair_value(res).reshape(b.M, b.C)
            _store_pair(y, F.relu(o) if relu else o)
        elif k == "maxpool_split":
            _, src, dst, n, h, w, c, kk, s, p = op
            v = _pair_value(src).reshape(n, h, w, c).permute(0, 3, 1, 2)
            _store_pair(dst, F.max_pool2d(v, kk, s, p).permute(0, 2, 3, 1).contiguous())
        elif k == "maxpool_bwd_split":
            _, xx, dy, dx, n, h, w, c, kk, s, p = op
            v = _pair_value(xx).reshape(n, h, w, c).permute(0, 3, 1, 2)
            oh, ow = (h + 2 * p - kk) // s + 1, (w + 2 * p - kk) // s + 1
            g = _first_max_pool_bwd(v, dy.float().reshape(n, oh, ow, c).permute(0, 3, 1, 2), kk, s, p)
            dx.copy_(g.permute(0, 2, 3, 1).half().reshape(dx.shape))
        elif k == "final_fwd_split":
            _, y5, logits = op
            yv = (y5[0].double() + y5[1].double()).permute(0, 3, 1, 2)
            logits.copy_(F.conv2d(yv, P["final.weight"].double(), P["final.bias"].double()).float())
        elif k == "wgrad":
            _, u, dy = op
            emulate.run_wgrad(u.wdesc, dy.data_ptr() + 2 * u.out_offset, u.dw_packed)
        else:
            emulate.run_train_ops(eng, [op], x=x, dlogits=dlogits)


def _rel(a, b):
    return ((a.double() - b.double()).pow(2).sum().sqrt() / b.double().pow(2).sum().sqrt().clamp_min(1e-30)).item()


def _plans(C, B=2, S=64):
    sd0 = {k[7:]: v.clone() for k, v in synth.make_state_dict(C, seed=0).items()}
    x = synth.normalize_tiles(synth.make_tiles_u8(B, S, seed=1))
    out = {}
    for precision in TRAIN_PRECISIONS:
        params = {k: v.clone() for k, v in sd0.items()}
        out[precision] = (params, UNetTrainEngine(params, C, B, S, S, device="cpu", plan_only=True, loss_scale=1024.0, precision=precision))
    return sd0, x, out


@pytest.mark.parametrize("classes", [2, 6])
def test_strict_plan_logits_match_oracle_train_forward(classes):
    sd0, x, plans = _plans(classes)
    sd = {k: v.clone() for k, v in sd0.items()}
    with torch.no_grad():
        ref = unet_oracle.unet_forward_train(sd, x)
    params, eng = plans["strict"]
    run_strict_train_ops(eng, eng.fwd_ops, x=x)
    strict = _rel(eng.logits, ref)
    fparams, feng = plans["fast"]
    emulate.run_train_ops(feng, feng.fwd_ops, x=x)
    fast = _rel(feng.logits, ref)
    print("%d classes, 2x64^2 train-mode logits vs the oracle, rel-L2: strict %.2e, fast %.2e" % (classes, strict, fast))
    assert strict <= 1e-5
    # running statistics follow torch's momentum / unbiased-variance update
    for name in [k[:-len(".running_mean")] for k in sd if k.endswith(".running_mean")]:
        assert _rel(params[name + ".running_mean"], sd[name + ".running_mean"]) <= 1e-5, name
        assert _rel(params[name + ".running_var"], sd[name + ".running_var"]) <= 1e-5, name
        assert int(params[name + ".num_batches_tracked"]) == int(sd0[name + ".num_batches_tracked"]) + 1, name


def test_strict_descriptors_are_split_forward_and_single_plane_backward():
    _, _, plans = _plans(2)
    params, eng = plans["strict"]
    run_strict_train_ops(eng, [("pack_all",)])
    assert len(eng.units) == len(eng.exponents) == len(eng.split_pack_list)
    for (name, u), (wname, _m, dst, scale, _single) in zip(eng.units.items(), eng.split_pack_list):
        d = u.desc
        assert d.split == 1 and wname == u.wname, name
        assert d.acc_scale == 2.0 ** -eng.exponents[name] and scale == 2.0 ** eng.exponents[name], name
        assert d.weights == dst.data_ptr() and dst.shape[0] == 2, name
        assert d.out_plane > 0 and d.out_plane % 8 == 0 and not d.residual and not d.stats, name
        for i in range(d.nsrc):
            assert d.srcs[i].plane > 0 and d.srcs[i].plane % 8 == 0, (name, i)
        # the plane stride is half the element count of the buffer the pointer lies in
        out_buf = [t for t in eng._keep if t.data_ptr() <= d.out < t.data_ptr() + t.numel() * 2 and t.dtype == torch.float16]
        assert len(out_buf) == 1 and out_buf[0].shape[0] == 2 and d.out_plane == out_buf[0].numel() // 2, name
        # the largest packed weight sits in [2^9, 2^10) after scaling (the overflow headroom of the plan)
        hi = dst[0].float().abs().max().item()
        assert 2.0 ** 9 <= hi <= 2.0 ** 10, (name, hi)
        w = u.wdesc
        assert w.split == 0 and w.acc_scale == 1.0 and w.kchunk == 0 and w.out_plane == 0 and w.out == d.out, name
        assert all(w.srcs[i].plane == 0 and w.srcs[i].ptr == d.srcs[i].ptr for i in range(w.nsrc)), name
    dgrads = [op[1].desc for op in eng.bwd_ops if op[0] == "conv"]
    assert len(dgrads) == 63
    for d in dgrads:
        assert d.split == 0 and all(d.srcs[i].plane == 0 for i in range(d.nsrc))
    # the backward reads single fp16 views: hi planes of the saved activations, no mask re-derived from single-plane z
    kinds = {op[0] for op in eng.fwd_ops}
    assert kinds == {"pack_all", "prepass_split", "conv", "bn_stats_split", "bn_apply_split", "maxpool_split", "final_fwd_split"}
    for op in eng.bwd_ops:
        if op[0] == "bn_bwd":
            assert op[3] is None or op[3].dim() == 4
            assert op[1].z.dim() == 4 and getattr(op[1], "plain_relu_y", None) is None
    # the fast plan is untouched: no split descriptor, no split op
    _, feng = plans["fast"]
    assert all(u.desc.split == 0 and u.wdesc is u.desc for u in feng.units.values())
    assert not feng.split_pack_list and {op[0] for op in feng.fwd_ops} == {"pack_all", "prepass", "conv", "bn_stats", "bn_finalize", "bn_apply",
                                                                          "maxpool", "final_fwd"}


def test_strict_plan_backward_reaches_every_parameter():
    """The whole strict step (forward, then the backward reading hi planes) replays through the emulation: finite gradients for
    all 168 trained tensors."""
    sd0, x, plans = _plans(2)
    params, eng = plans["strict"]
    run_strict_train_ops(eng, eng.fwd_ops, x=x)
    g = torch.Generator().manual_seed(3)
    dl = torch.randn((2, 2, 64, 64), generator=g) * 1e-3
    run_strict_train_ops(eng, eng.bwd_ops, dlogits=dl)
    assert len(eng.grads) == 168 and all(torch.isfinite(v).all() for v in eng.grads.values())
    assert all(float(v.abs().sum()) > 0 for k, v in eng.grads.items())


def test_train_precision_selection(monkeypatch):
    monkeypatch.delenv("RSB_TRAIN_PRECISION", raising=False)
    assert default_train_precision() == "fast"
    monkeypatch.setenv("RSB_TRAIN_PRECISION", "STRICT")
    assert default_train_precision() == "strict"
    sd = {k[7:]: v for k, v in synth.make_state_dict(2, seed=0).items()}
    assert UNetTrainEngine(sd, 2, 1, 64, 64, device="cpu", plan_only=True).strict
    monkeypatch.setenv("RSB_TRAIN_PRECISION", "double")
    with pytest.raises(ValueError, match="RSB_TRAIN_PRECISION"):
        default_train_precision()
    with pytest.raises(ValueError, match="RSB_TRAIN_PRECISION"):
        UNetTrainEngine(sd, 2, 1, 64, 64, device="cpu", plan_only=True)
    with pytest.raises(ValueError, match="precision"):
        UNetTrainEngine(sd, 2, 1, 64, 64, device="cpu", plan_only=True, precision="half")
    from robosat_b200.unet import UNet

    net = UNet(2, pretrained=False)
    assert net.train_precision is None and net.precision is None


def test_new_entry_points_validate_then_need_a_device():
    """Argument errors are RSB_E_INVALID on any host; valid arguments fail with RSB_E_NODEVICE without a device (no CPU path)."""
    import ctypes

    from robosat_b200 import _lib

    if torch.cuda.is_available():
        pytest.skip("GPU present")
    lib = _lib.load()
    buf = torch.zeros(1 << 16, dtype=torch.float32)
    a = buf.data_ptr()
    calls = {
        "rsb_pack_weights_split": (lambda ok: lib.rsb_pack_weights_split(a, a, a, 64, 64 if ok else 65, 2.0, a, None)),
        "rsb_pack_weights1_split": (lambda ok: lib.rsb_pack_weights1_split(a, a, a, 64, 64 if ok else 60, 2.0, a, None)),
        "rsb_bn_stats_finalize_split": (lambda ok: lib.rsb_bn_stats_finalize_split(a, 1024, a, a, a, a, a, a, a, a, a, a, 16, 64 if ok else 60,
                                                                                   1e-5, 0.1, None, None)),
        "rsb_bn_stats_finalize_split_chained": (lambda ok: lib.rsb_bn_stats_finalize_split_chained(a, 1024 if ok else 1023, a, a, a, a, a, a, a, a,
                                                                                                   a, a, 16, 64, 1e-5, 0.1, a, None)),
        "rsb_bn_apply_split": (lambda ok: lib.rsb_bn_apply_split(a, 1024, a, a, None, 0, a, 1024 if ok else 0, 16, 64, 1, None)),
        "rsb_bn_apply_split_chained": (lambda ok: lib.rsb_bn_apply_split_chained(a, 1024, a, a, a if ok else None, 1024, a, 1024, 16, 64 if ok else 12,
                                                                                 1, None)),
        "rsb_maxpool_backward_split": (lambda ok: lib.rsb_maxpool_backward_split(a, 1024, a, a, a if ok else None, 1, 4, 4, 64, 2, 2, 0, None)),
        "rsb_final_forward_split": (lambda ok: lib.rsb_final_forward_split(a, 1024, a, a, None, a, 1, 16, 2 if ok else 9, None)),
    }
    for name, call in calls.items():
        assert call(False) == -1, name
        assert call(True) == -3, (name, _lib.last_error())
