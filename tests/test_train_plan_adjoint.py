"""Every backward descriptor of the training plan is the exact adjoint of its forward descriptor (CPU, emulated).

For each conv unit of a 64x64 plan_only UNetTrainEngine, with random fp16 activations / gradients and random fp32 weights,
on a copy of the forward descriptor without ReLU, statistics or residual (a linear map F(x; w)):
  - input gradient:  <F(x), dy> == sum over the unit's backward-conv launches s (one per concat source) of <x_s, dgrad_s(dy)>,
    the launches run without their fan-in residual. Covers map_conv_dgrad (padded Cout included), map_s2_dgrad and the per-source
    split of map_up_dgrad, and the output addressing of every backward conv (phases, strides, offsets into padded buffers).
  - weight gradient: <F(x; w), dy> == <w, unpack(wgrad(dy))> with w packed by the unit's own forward map. Covers the scatter-back
    of every forward map (stem window, dec5 window, parity views, summed upsample taps).
x is random only where the backward launches write (so zero in pad columns and on the odd pixels of a stride-2 downsample).

Both sides are float64 sums of products of fp16 values; the only roundings are the fp16 stores of F(x) / dgrad(dy) and of the
packed weights (relative 2^-11 each, independent signs), so each side is within ~2^-11 * ||terms||_2 of the exact adjoint
pairing. The bound is 1e-3 * (||F(x) * dy||_2 + ||other side's terms||_2). An index-map error moves whole taps: the difference
is then of the order of the norms themselves.
"""

import numpy as np
import torch

import emulate
from robosat_b200 import synth
from robosat_b200._lib import ConvDesc
from robosat_b200.train_engine import UNetTrainEngine

from test_train_ops_gpu import AddressMap, view

REL = 1e-3


def _copy(desc, linear):
    d = ConvDesc.from_buffer_copy(desc)
    d.residual = None
    if linear:
        d.relu, d.stats, d.stats_bytes = 0, None, 0
    return d


def _pack(eng, wname, w):
    """fp32 OIHW w -> every packed fp16 layout of `wname` (forward and backward maps), as the pack_all op does"""
    src = w.reshape(-1)
    for name, m, dst, _c, _o in eng.pack_list:
        if name == wname:
            mm = m.long()
            dst.copy_(torch.where(mm >= 0, src[mm.clamp_min(0)], torch.zeros(())).sum(1).half())


def _pairing(a, b):
    """(<a, b> in float64, ||a * b||_2)"""
    p = a.double() * b.double()
    return float(p.sum()), float(p.pow(2).sum().sqrt())


def test_backward_descriptors_are_adjoints_of_the_forward():
    C, B, S = 2, 2, 64
    sd = {k[7:]: v for k, v in synth.make_state_dict(C, seed=0).items()}
    eng = UNetTrainEngine(sd, C, B, S, S, device="cpu", plan_only=True, loss_scale=1024.0)
    bufs = [("keep%d" % i, t) for i, t in enumerate(eng._keep)]
    amap = AddressMap(bufs)
    g = torch.Generator().manual_seed(11)
    wgrad_dy = {op[1].name: op[2] for op in eng.bwd_ops if op[0] == "wgrad"}
    checked = {"input": 0, "weight": 0, "dgrad_launches": 0}
    worst = []
    for name, u in eng.units.items():
        fwd = _copy(u.desc, linear=True)
        dgrads = [_copy(op[1].desc, linear=False) for op in eng.bwd_ops if op[0] == "conv" and op[1].name.startswith(name + ".dgrad")]
        w = torch.randn(u.wshape, generator=g) * (2.0 / np.prod(u.wshape[1:])) ** 0.5
        _pack(eng, u.wname, w)

        # x: the distinct forward source buffers, in order, paired with the backward launches (one per concat source)
        src_bufs = list(dict.fromkeys(amap.find(fwd.srcs[i].ptr)[0] for i in range(fwd.nsrc)))
        for bi in src_bufs:
            bufs[bi][1].zero_()
        x_regions = []
        if dgrads:
            assert len(dgrads) == len(src_bufs), name
            for bi, dd in zip(src_bufs, dgrads):
                r = amap.conv_out(dd)
                assert bufs[r[0]][1].shape == bufs[bi][1].shape, name
                xr = (bi,) + r[1:]
                view(bufs, xr).copy_(torch.randn(xr[1], generator=g).half())
                x_regions.append((xr, r))
        else:  # the stem: the input image has no gradient; any x serves the weight check
            assert name == "stem"
            for bi in src_bufs:
                bufs[bi][1].copy_(torch.randn(bufs[bi][1].shape, generator=g).half())

        # dy: random in the forward output region of the gradient buffer the backward reads (same layout as the output)
        out_r = amap.conv_out(fwd)
        dy_t = wgrad_dy[name]
        dy_i, dy_off = amap.find(dy_t.data_ptr())
        assert dy_off == 0 and dy_t.shape == bufs[out_r[0]][1].shape, name
        dy_t.zero_()
        dy_r = (dy_i,) + out_r[1:]
        view(bufs, dy_r).copy_(torch.randn(out_r[1], generator=g).half())

        emulate.run_desc(fwd)
        lhs, lhs_n = _pairing(view(bufs, out_r), view(bufs, dy_r))

        if dgrads:
            rhs, rhs_n = 0.0, 0.0
            for dd, (xr, r) in zip(dgrads, x_regions):
                for s in range(dd.nsrc):
                    assert amap.find(dd.srcs[s].ptr)[0] == dy_i, name  # every backward launch reads this unit's dy
                emulate.run_desc(dd)
                p, n2 = _pairing(view(bufs, xr), view(bufs, r))
                rhs, rhs_n = rhs + p, (rhs_n ** 2 + n2 ** 2) ** 0.5
            ratio = abs(lhs - rhs) / (REL * (lhs_n + rhs_n))
            worst.append((ratio, name, "input"))
            assert ratio <= 1.0, "%s: <F(x), dy> = %.6g but the backward launches give %.6g (scale %.3g)" % (name, lhs, rhs, lhs_n + rhs_n)
            checked["input"] += 1
            checked["dgrad_launches"] += len(dgrads)

        dw = torch.zeros(u.dw_packed.shape, dtype=torch.float32)
        emulate.run_wgrad(u.desc, dy_t.data_ptr() + 2 * u.out_offset, dw)
        gw = torch.zeros(w.numel(), dtype=torch.float64)
        mm = u.fwd_map.long()
        for j in range(4):
            sel = mm[:, j] >= 0
            gw.index_add_(0, mm[sel, j], dw[sel].double())
        rhs_w, rhs_wn = _pairing(w.reshape(-1), gw)
        ratio = abs(lhs - rhs_w) / (REL * (lhs_n + rhs_wn))
        worst.append((ratio, name, "weight"))
        assert ratio <= 1.0, "%s: <F(x; w), dy> = %.6g but <w, unpack(wgrad(dy))> = %.6g (scale %.3g)" % (name, lhs, rhs_w, lhs_n + rhs_wn)
        checked["weight"] += 1

    print("adjoint checks %s, worst error / allowed: %s" % (checked, sorted(worst)[-3:]))
    assert checked == {"input": len(eng.units) - 1, "weight": len(eng.units), "dgrad_launches": 63}
