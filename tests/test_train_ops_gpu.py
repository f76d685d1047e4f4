"""Every launch of one UNetTrainEngine step (forward + backward, ~420 ops) against the CPU emulation of that one op.

The GPU engine runs kernel by kernel; a CPU `plan_only` engine built from the same arguments (identical buffer list) is the
mirror and replays the op with tests/emulate.py on the same inputs. Per op:
  1. snapshot every engine buffer, the parameters and the flat gradient buffer (the int32 index maps never change),
  2. fill with NaN what the op must write in full without reading it (and the conv's `stats` rows),
  3. run the GPU op and the emulation,
  4. compare the declared outputs within an error model (below),
  5. require everything else -- other buffers, parameters, the rest of the gradient buffer, pad columns -- to be bit-identical
     to the snapshot (chained BatchNorm launches must also leave their accumulators zeroed),
  6. copy the GPU outputs into the mirror, so every op is judged on its own inputs.

Error model (u = 2^-24, the fp32 unit roundoff; ulp = fp16 spacing at the larger of the two values):
  - bit-identical: single-source weight packing, prepass, maxpool, relu_bwd, g_out, non-overlapping maxpool_bwd, zero_grads
  - <= 1 ulp: pre-summed (upsample) weight packing and overlapping maxpool_bwd windows (a sum of <= 4 fp16 values in another order)
  - bn_apply: 1 ulp + 2u (|z*scale| + |shift| + |res|): the kernel fuses z*scale + shift into one fma, the emulation rounds twice
  - fp16 conv outputs: 1 ulp + 2(K+1)u * mag, mag = sum_k |a_k w_k| bounded per segment by Cauchy-Schwarz; any order of a K-term
    fp32 sum is within K*u*mag of the exact sum, truncating tensor-core adds within 2u per add, and both sides round once more
  - reductions inside a launch (BatchNorm sums, final 1x1 gradients, weight gradients) are fp32 chains of at most n terms
    (n = rows / pixels reduced), so each sum is within n*u * (sum of magnitudes) of the exact one; the fp64 emulation is exact
    at that scale. BatchNorm statistics, dz, dgamma / dbeta propagate that bound through their formulas.
"""

import bisect
import os

import numpy as np
import pytest
import torch

import emulate
from robosat_b200 import synth, train_engine
from robosat_b200.train_engine import UNetTrainEngine

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
_INT = {torch.float16: torch.int16, torch.float32: torch.int32, torch.float64: torch.int64}


def _bits(t):
    return t.view(_INT.get(t.dtype, t.dtype))


def ulp16(x):
    """spacing of fp16 at |x| (float64 tensor in, float64 out; subnormal spacing 2^-24 below 2^-14)"""
    _, e = torch.frexp(x.abs().float())
    return torch.ldexp(torch.ones_like(x, dtype=torch.float64), (e.long() - 11).clamp_min(-24))


# --------------------------------------------------------------------------------------------------
# buffers and regions
# --------------------------------------------------------------------------------------------------
def engine_buffers(eng):
    """the engine's state in a fixed order: its buffers (without the constant int32 index maps), the flat gradient
    buffer and the parameters. A GPU engine and a plan_only engine built from the same arguments give matching lists."""
    eng._grad("final.bias")
    bufs = [("keep%d" % i, t) for i, t in enumerate(eng._keep) if t.dtype != torch.int32]
    bufs.append(("grads", eng._grads_flat))
    bufs += [("param:" + k, v) for k, v in eng.params.items()]
    return bufs


class AddressMap:
    """device address -> (buffer index, element offset), by interval lookup over the buffer list"""

    def __init__(self, bufs):
        self.ranges = sorted((t.data_ptr(), t.data_ptr() + t.numel() * t.element_size(), i) for i, (_, t) in enumerate(bufs))
        self.starts = [r[0] for r in self.ranges]
        self.bufs = bufs

    def find(self, ptr):
        j = bisect.bisect_right(self.starts, ptr) - 1
        assert j >= 0 and ptr < self.ranges[j][1], "address %#x is in no engine buffer" % ptr
        lo, _, i = self.ranges[j]
        item = self.bufs[i][1].element_size()
        assert (ptr - lo) % item == 0
        return i, (ptr - lo) // item

    def region(self, t):
        i, off = self.find(t.data_ptr())
        return (i, tuple(t.shape), tuple(t.stride()), off)

    def conv_out(self, d):
        """what a conv descriptor writes: out + n*pitch_n + (h*sy+a)*pitch_h + (w*sx+b)*pitch_w + c, phases (a, b)"""
        i, off = self.find(d.out)
        size = (d.Nt, d.Ht, d.Wt, d.Cout)
        stride = (d.out_pitch_n, d.out_sy * d.out_pitch_h, d.out_sx * d.out_pitch_w, 1)
        if d.phases == 4:
            size, stride = (2, 2) + size, (d.out_pitch_h, d.out_pitch_w) + stride
        return (i, size, stride, off)


def view(bufs, region):
    i, size, stride, off = region
    return bufs[i][1].reshape(-1).as_strided(size, stride, off)


# --------------------------------------------------------------------------------------------------
# what each op writes, and how its result is judged
# --------------------------------------------------------------------------------------------------
class Out:
    def __init__(self, label, region, check, poison, ctx=None):
        self.label, self.region, self.check, self.poison, self.ctx = label, region, check, poison, ctx


def _conv_mag(d):
    """per output element, an upper bound of sum_k |a_k w_k| (Cauchy-Schwarz per segment): float64 [phases, Nt, Ht, Wt, Cout]"""
    K = 64 * sum(d.segs[i].cblocks for i in range(d.nseg))
    wts = emulate._view(d.weights, (d.phases * d.Cout, K), (K, 1)).astype(np.float64)
    mags = []
    for phase in range(d.phases):
        m = np.zeros((d.Nt, d.Ht, d.Wt, d.Cout))
        k0 = 0
        for si in range(d.nseg):
            a = emulate._gather_segment(d, d.segs[si], phase).astype(np.float64)
            w = wts[phase * d.Cout:(phase + 1) * d.Cout, k0:k0 + a.shape[-1]]
            m += np.sqrt((a * a).sum(-1))[..., None] * np.sqrt((w * w).sum(1))
            k0 += a.shape[-1]
        mags.append(m)
    return np.stack(mags), K


def _wgrad_mag(d, dy_ptr):
    """per packed gradient element, an upper bound of sum_p |dy_p a_p| (Cauchy-Schwarz over the pixels): float64 [phases*Cout, K]"""
    K = 64 * sum(d.segs[i].cblocks for i in range(d.nseg))
    out = np.zeros((d.phases * d.Cout, K))
    for phase in range(d.phases):
        pa, pb = phase >> 1, phase & 1
        dyv = emulate._view(dy_ptr + 2 * (pa * d.out_pitch_h + pb * d.out_pitch_w), (d.Nt, d.Ht, d.Wt, d.Cout),
                            (d.out_pitch_n, d.out_sy * d.out_pitch_h, d.out_sx * d.out_pitch_w, 1)).astype(np.float64)
        ndy = np.sqrt((dyv * dyv).reshape(-1, d.Cout).sum(0))
        k0 = 0
        for si in range(d.nseg):
            a = emulate._gather_segment(d, d.segs[si], phase).astype(np.float64)
            na = np.sqrt((a * a).reshape(-1, a.shape[-1]).sum(0))
            out[phase * d.Cout:(phase + 1) * d.Cout, k0:k0 + a.shape[-1]] = ndy[:, None] * na[None, :]
            k0 += a.shape[-1]
    return out


def declared(amap, gpu, cpu, cbufs, dlogits, gop, cop):
    """(outputs, scratch regions, accumulator regions that must be zero afterwards) of one GPU op; tolerance inputs are taken
    from the mirror, whose state equals the GPU's before the op"""
    k = gop[0]
    outs, scratch, zeroed = [], [], []
    P = cpu.params

    def reg(t):
        return amap.region(t)

    def sums_regions(b):
        i, off = amap.find(b.sums.data_ptr())
        slots = (i, (16 * b.C + 2,), (1,), off)                      # 8 slots x {sum, sum of squares} x C, arrival counter, pad
        coef = (i, (-(-3 * b.C // 2),), (1,), off + 16 * b.C + 2)  # 3*C fp32 backward coefficients
        return slots, coef

    if k == "conv":
        d, dc = gop[1].desc, cop[1].desc
        region = amap.conv_out(d)
        in_place = bool(d.residual) and d.residual == d.out  # fan-in sums accumulate into the output itself
        mag, K = _conv_mag(dc)
        res = np.zeros_like(mag)
        if d.residual:  # addressed like the output
            ri, roff = amap.find(d.residual)
            res = np.abs(view(cbufs, (ri,) + region[1:3] + (roff,)).double().numpy()).reshape(mag.shape)
        outs.append(Out("out", region, "conv", not in_place, (mag, K, res)))
        if d.stats:
            i, off = amap.find(d.stats)
            rows = 4 * (-(-d.Wt // d.TW)) * (-(-d.Ht // d.TH)) * (-(-d.Nt // d.TN))
            outs.append(Out("stats", (i, (rows, 2, d.Cout), (2 * d.Cout, d.Cout, 1), off), "stats", True, region))
    elif k == "pack_all":
        for (wname, _, dst, _, _), (_, m, _, _, _) in zip(gpu.pack_list, cpu.pack_list):
            single = bool((m[:, 1:] < 0).all())
            outs.append(Out("pack " + wname, reg(dst), "exact" if single else "ulp", True))
    elif k == "prepass":
        outs.append(Out("s2d", reg(gpu.s2d), "exact", True))
    elif k == "maxpool":
        outs.append(Out("dst", reg(gop[2]), "exact", True))
    elif k == "maxpool_bwd":
        kk, s = gop[8], gop[9]
        outs.append(Out("dx", reg(gop[3]), "exact" if kk == s else "ulp", True))
    elif k == "relu_bwd":
        _, a, b2, y, out = gop
        outs.append(Out("out", reg(out), "exact", out is not a and out is not b2))
    elif k == "bn_stats":
        b, bc = gop[1], cop[1]
        pf = b.prefix
        z = bc.z.reshape(bc.M, bc.C).double()
        ctx = dict(M=bc.M, sabs=z.abs().sum(0), ssq=(z * z).sum(0), mean=z.mean(0), var=(z * z).mean(0) - z.mean(0) ** 2,
                   gamma=P[pf + ".weight"].double(), beta=P[pf + ".bias"].double(), rm=P[pf + ".running_mean"].double())
        for nm, t, poison in (("mean", b.mean, True), ("invstd", b.invstd, True), ("scale", b.scale, True), ("shift", b.shift, True),
                              ("running_mean", gpu.params[pf + ".running_mean"], False),
                              ("running_var", gpu.params[pf + ".running_var"], False)):
            outs.append(Out(nm, reg(t), "bn_" + nm, poison, ctx))
        outs.append(Out("num_batches_tracked", reg(gpu.params[pf + ".num_batches_tracked"]), "exact", False))
        slots, _ = sums_regions(b)
        (zeroed if train_engine.BN_CHAINED else scratch).append(slots)
    elif k == "bn_finalize":
        pass  # folded into the bn_stats launch: must write nothing
    elif k == "bn_apply":
        _, b, res, y, relu = gop
        bc = cop[1]
        mag = (bc.z.reshape(bc.M, bc.C).double() * bc.scale.double()).abs() + bc.shift.double().abs()
        if res is not None:
            mag = mag + cop[2].reshape(bc.M, bc.C).double().abs()
        outs.append(Out("y", reg(y), "bn_apply", True, mag.reshape(tuple(y.shape))))
    elif k == "bn_bwd":
        _, b, dy, y, dz, g = gop
        _, bc, dyc, yc, _, _ = cop
        pf = b.prefix
        gg = dyc.reshape(bc.M, bc.C).double()
        if yc is not None:
            gg = gg * (yc.reshape(bc.M, bc.C).double() > 0)
        zz = bc.z.reshape(bc.M, bc.C).double()
        mu, inv = bc.mean.double(), bc.invstd.double()
        zhat = (zz - mu) * inv
        A = (P[pf + ".weight"].double() * inv).abs()
        ctx = dict(M=bc.M, g=gg, zhat=zhat, A=A, inv=inv, mu=mu, ls=cpu.loss_scale, sabs_g=gg.abs().sum(0),
                   sabs_gz=(gg * zz).abs().sum(0), sabs_gzh=(gg * zhat).abs().sum(0), mgz=(gg * zhat).mean(0), mg=gg.mean(0))
        outs.append(Out("dz", reg(dz), "bn_dz", dz is not dy, ctx))
        if g is not None:
            outs.append(Out("g_out", reg(g), "exact", g is not dy))
        outs.append(Out("dgamma", reg(gpu.grads[pf + ".weight"]), "bn_dgamma", True, ctx))
        outs.append(Out("dbeta", reg(gpu.grads[pf + ".bias"]), "bn_dbeta", True, ctx))
        slots, coef = sums_regions(b)
        scratch.append(coef)
        (zeroed if train_engine.BN_CHAINED else scratch).append(slots)
    elif k == "wgrad":
        u, uc = gop[1], cop[1]
        d = uc.desc
        mag = _wgrad_mag(d, cop[2].data_ptr() + 2 * uc.out_offset)
        outs.append(Out("dw_packed", reg(u.dw_packed), "wgrad", True, (mag.reshape(-1), d.Nt * d.Ht * d.Wt)))
    elif k == "unpack_all":
        deterministic = os.environ.get("RSB_WGRAD_DETERMINISTIC", "1") != "0"
        flat = torch.zeros_like(cpu._grads_flat, dtype=torch.float64)
        for dwp, m, wname, _c, _o in cpu.unpack_list:
            mm = m.long()
            for j in range(4):
                sel = mm[:, j] >= 0
                flat.index_add_(0, mm[sel, j] + cpu._grad_offset[wname], dwp[sel].double().abs() / cpu.loss_scale)
        for wname in dict.fromkeys(w for _, _, w, _, _ in cpu.unpack_list):
            o = cpu._grad_offset[wname]
            n = cpu.grads[wname].numel()
            outs.append(Out("grad " + wname, reg(gpu.grads[wname]), "unpack", deterministic, flat[o:o + n].reshape(cpu.grads[wname].shape)))
    elif k == "zero_grads":
        outs.append(Out("grads", reg(gpu._grads_flat), "exact", True))
    elif k == "final_fwd":
        y5 = cop[1].double().reshape(-1, 32)
        w, bb = P["final.weight"].double().reshape(cpu.C, 32), P["final.bias"].double()
        mag = (y5.abs() @ w.abs().t() + bb.abs()).reshape(cpu.N, cpu.H, cpu.W, cpu.C).permute(0, 3, 1, 2)
        outs.append(Out("logits", reg(gop[2]), "fp32sum", True, (mag, 33)))
    elif k == "final_bwd":
        dl = dlogits.double().permute(0, 2, 3, 1).reshape(-1, cpu.C)
        y5 = cop[1].double().reshape(-1, 32)
        w = P["final.weight"].double().reshape(cpu.C, 32)
        mag_dx = ((dl.abs() * cpu.loss_scale) @ w.abs()).reshape(tuple(gop[2].shape))
        outs.append(Out("d_y5", reg(gop[2]), "fp16sum", True, (mag_dx, cpu.C + 1)))
        npx = y5.shape[0]
        outs.append(Out("final.weight grad", reg(gpu.grads["final.weight"]), "fp32sum", True,
                        ((dl.abs().t() @ y5.abs()).reshape(cpu.C, 32, 1, 1), npx + 1)))
        outs.append(Out("final.bias grad", reg(gpu.grads["final.bias"]), "fp32sum", True, (dl.abs().sum(0), npx + 1)))
        i, off = amap.find(gpu.final_acc.data_ptr())
        scratch.append((i, (gpu.final_acc.numel(),), (1,), off))
    else:  # pragma: no cover
        raise AssertionError(k)
    return outs, scratch, zeroed


def judge(o, got, ref):
    """worst error / allowed error of one output (> 1 fails; NaN / inf count as failures)"""
    c = o.check
    if c == "exact":
        return 0.0 if torch.equal(_bits(got.contiguous()), _bits(ref.contiguous())) else float("inf")
    a, b = got.double(), ref.double()
    err = (a - b).abs()
    big = torch.maximum(a.abs(), b.abs())
    if c == "ulp":
        tol = ulp16(big)
    elif c == "bn_apply":
        tol = ulp16(big) + 2 * U * o.ctx
    elif c == "conv":
        mag, K, res = o.ctx
        tol = ulp16(big) + torch.from_numpy(2 * (K + 1) * U * mag.reshape(tuple(got.shape)) + 2 * U * res.reshape(tuple(got.shape)))
    elif c == "fp16sum":
        mag, n = o.ctx
        tol = ulp16(big) + 2 * n * U * mag
    elif c == "fp32sum":
        mag, n = o.ctx
        tol = 2 * n * U * mag + 2 * U * big
    elif c == "wgrad":
        mag, n = o.ctx
        tol = 2 * (n + 1) * U * torch.from_numpy(mag) + 2 * U * big
    elif c == "unpack":
        tol = 8 * U * o.ctx.reshape(tuple(got.shape)) + 2 * U * big
    elif c.startswith("bn_"):
        tol = _bn_tol(c, o.ctx, big)
    else:  # pragma: no cover
        raise AssertionError(c)
    ok = err <= tol
    if bool(ok.all()):
        return float((err / tol.clamp_min(1e-300)).max()) if err.numel() else 0.0
    return float("inf") if not bool(torch.isfinite(a).all()) else float((err / tol.clamp_min(1e-300)).max())


def _bn_tol(c, x, big):
    M = x["M"]
    gM = (M + 32) * U  # an fp32 chain over at most M rows (+ the 32-row partials of the conv epilogue)
    if c in ("bn_mean", "bn_invstd", "bn_scale", "bn_shift", "bn_running_mean", "bn_running_var"):
        dmean = gM * x["sabs"] / M + U * x["mean"].abs()
        dvar = gM * x["ssq"] / M + 2 * x["mean"].abs() * dmean + 4 * U * x["ssq"] / M
        var = x["var"].clamp_min(0)
        inv = 1.0 / torch.sqrt(var + 1e-5)
        dinv = 0.5 * inv ** 3 * dvar + 2 * U * inv
        if c == "bn_mean":
            return dmean + 2 * U * big
        if c == "bn_invstd":
            return dinv + 2 * U * big
        if c == "bn_scale":
            return x["gamma"].abs() * dinv + 2 * U * big
        if c == "bn_shift":
            sc = x["gamma"].abs() * inv
            return dmean * sc + x["mean"].abs() * x["gamma"].abs() * dinv + 4 * U * (x["beta"].abs() + x["mean"].abs() * sc) + 2 * U * big
        if c == "bn_running_mean":
            return 0.1 * dmean + 4 * U * (x["rm"].abs() + x["mean"].abs()) + 2 * U * big
        return 0.1 * dvar * M / (M - 1) + 4 * U * big + 4 * U * var
    g, zhat, A, inv, mu, ls = x["g"], x["zhat"], x["A"], x["inv"], x["mu"], x["ls"]
    if c == "bn_dbeta":
        return gM * x["sabs_g"] / ls + 2 * U * big
    if c == "bn_dgamma":
        # the kernel sums g*z and g and forms (sum gz - mu sum g) * invstd; the emulation sums g * fp32 zhat
        return (gM * inv * (x["sabs_gz"] + mu.abs() * x["sabs_g"]) + 4 * U * x["sabs_gzh"]) / ls + 2 * U * big
    # dz = gamma*invstd*(g - mean(g) - zhat*mean(g*zhat)): both sides evaluate ~4 fp32 operations per element on the same
    # inputs; the kernel's means carry the reduction bound
    dmg = gM * x["sabs_g"] / M
    dmgz = gM * inv * (x["sabs_gz"] + mu.abs() * x["sabs_g"]) / M + U * x["mgz"].abs()
    terms = A * (g.abs() + x["mg"].abs() + zhat.abs() * x["mgz"].abs())
    return (ulp16(big.reshape(g.shape)) + 8 * U * terms + A * (dmg + zhat.abs() * dmgz)).reshape(big.shape)


# --------------------------------------------------------------------------------------------------
# the replay
# --------------------------------------------------------------------------------------------------
def _paired_ops(gpu_ops, cpu_ops):
    """GPU op -> the emulator ops it corresponds to (bn_stats = stats + finalize; bn_finalize is a no-op on the GPU)"""
    assert [o[0] for o in gpu_ops] == [o[0] for o in cpu_ops]
    pairs = []
    for i, (g, c) in enumerate(zip(gpu_ops, cpu_ops)):
        if g[0] == "bn_stats":
            assert cpu_ops[i + 1][0] == "bn_finalize" and cpu_ops[i + 1][1] is c[1]
            pairs.append((g, c, [c, cpu_ops[i + 1]]))
        elif g[0] == "bn_finalize":
            pairs.append((g, c, []))
        else:
            pairs.append((g, c, [c]))
    return pairs


def _op_name(op):
    k = op[0]
    if k == "conv":
        return op[1].name
    if k in ("wgrad", "bn_stats", "bn_finalize", "bn_apply", "bn_bwd"):
        return op[1].name
    return k


def replay_step(gpu, cpu, x, dlogits, run_gpu, sync, table, lists=("fwd", "bwd")):
    """replay the op lists `lists` of `gpu` op by op against the emulation on `cpu`; returns (ops checked, failures)"""
    gbufs, cbufs = engine_buffers(gpu), engine_buffers(cpu)
    assert len(gbufs) == len(cbufs)
    for (gn, g), (cn, c) in zip(gbufs, cbufs):
        assert gn == cn and g.shape == c.shape and g.dtype == c.dtype, (gn, g.shape, c.shape)
    assert [t.shape for t in gpu._keep] == [t.shape for t in cpu._keep]
    amap, camap = AddressMap(gbufs), AddressMap(cbufs)
    xg, dlg = x.to(gpu.device), dlogits.to(gpu.device)
    failures, n = [], 0
    for phase in lists:
        gops, cops = getattr(gpu, phase + "_ops"), getattr(cpu, phase + "_ops")
        for idx, (gop, cop, emu) in enumerate(_paired_ops(gops, cops)):
            where = "%s op %d %s [%s]" % (phase, idx, gop[0], _op_name(gop))
            outs, scratch, zeroed = declared(amap, gpu, cpu, cbufs, dlogits, gop, cop)
            if gop[0] == "conv":  # the mirror's descriptor addresses the same buffers at the same offsets
                assert camap.conv_out(cop[1].desc)[:1] + camap.conv_out(cop[1].desc)[3:] == amap.conv_out(gop[1].desc)[:1] + amap.conv_out(gop[1].desc)[3:], where
            snap = [t.clone() for _, t in gbufs]
            for o in outs:
                if o.poison:
                    v = view(gbufs, o.region)
                    v.fill_(float("nan") if v.is_floating_point() else -1)
            run_gpu(gop, xg, dlg)
            sync()
            emulate.run_train_ops(cpu, emu, x=x, dlogits=dlogits)
            # declared outputs
            for o in outs:
                got = view(gbufs, o.region).cpu()
                if o.check == "stats":
                    z = view(gbufs, o.ctx).double().cpu().reshape(-1, got.shape[-1])  # the GPU's own z
                    tot = got.double().sum(0)
                    ok0 = (tot[0] - z.sum(0)).abs() <= 32 * U * z.abs().sum(0) * 2 + 1e-30
                    ok1 = (tot[1] - (z * z).sum(0)).abs() <= 33 * U * (z * z).sum(0) * 2 + 1e-30
                    r = 0.0 if bool(ok0.all() and ok1.all() and torch.isfinite(got).all()) else float("inf")
                else:
                    r = judge(o, got, view(cbufs, o.region))
                table.setdefault(gop[0] + ":" + o.check, [0.0, ""])
                if r > table[gop[0] + ":" + o.check][0]:
                    table[gop[0] + ":" + o.check] = [r, where + " " + o.label]
                if not r <= 1.0:
                    failures.append("%s: %s off by %.3g x the allowed error" % (where, o.label, r))
            # nothing else may change
            written = {}
            for reg in [o.region for o in outs] + scratch:
                m = written.get(reg[0])
                if m is None:
                    m = written[reg[0]] = torch.zeros(gbufs[reg[0]][1].numel(), dtype=torch.bool, device=gpu.device)
                m.as_strided(reg[1], reg[2], reg[3]).fill_(True)
            for bi, (bn, t) in enumerate(gbufs):
                cur, old = _bits(t.reshape(-1)), _bits(snap[bi].reshape(-1))
                if bi in written:
                    bad = int(((cur != old) & ~written[bi]).sum())
                else:
                    bad = 0 if torch.equal(cur, old) else int((cur != old).sum())
                if bad:
                    failures.append("%s: %d stray writes into %s" % (where, bad, bn))
            for reg in zeroed:
                if not bool((_bits(view(gbufs, reg)) == 0).all()):
                    failures.append("%s: BatchNorm accumulators not left zeroed" % where)
            # teacher forcing
            for o in outs:
                view(cbufs, o.region).copy_(view(gbufs, o.region).cpu())
            n += 1
            if len(failures) > 20:
                break
    return n, failures


def _make_engines(C, B, H, W, gpu_device):
    sd = {k[7:]: v for k, v in synth.make_state_dict(C, seed=0).items()}
    g = torch.Generator().manual_seed(7)
    x = synth.normalize_tiles(synth.make_tiles_u8(B, max(H, W), seed=1))[:, :, :H, :W].contiguous()
    dlogits = torch.randn((B, C, H, W), generator=g) * 1e-3
    cpu = UNetTrainEngine({k: v.clone() for k, v in sd.items()}, C, B, H, W, device="cpu", plan_only=True, loss_scale=1024.0)
    gpu = UNetTrainEngine({k: v.clone().to(gpu_device) for k, v in sd.items()}, C, B, H, W, device=gpu_device, loss_scale=1024.0)
    return gpu, cpu, x, dlogits


def _print_table(title, table):
    print("\n%s: worst error / allowed error per op kind and check" % title)
    for key in sorted(table):
        r, where = table[key]
        print("  %-28s %8.3g   %s" % (key, r, where))


@pytest.mark.parametrize("cfg", ["a", "b", "c"])
def test_every_train_launch_matches_its_emulation(cfg, cuda_device, monkeypatch):
    """(a) 2 classes, batch 2, 64x64 on the default paths (conv-epilogue statistics, chained BatchNorm, deterministic wgrad);
    (b) 6 classes, batch 3, 64x128 (odd batch, non-square, dec5 with more tiles than SMs) on the other paths (z reduction,
    unchained BatchNorm, fp32-atomic wgrad and scatter unpack);
    (c) the forward of (a) at 128x128: there the statistics of the stem and layer1 are folded by >= 8 blocks, so every one of
    the 8 accumulator slots of rsb_bn_partials_finalize is in use (at 64x64 no layer has enough partial rows)."""
    lists = ("fwd", "bwd")
    if cfg == "b":
        monkeypatch.setattr(train_engine, "CONV_STATS", False)
        monkeypatch.setattr(train_engine, "BN_CHAINED", False)
        monkeypatch.setenv("RSB_WGRAD_DETERMINISTIC", "0")
        C, B, H, W = 6, 3, 64, 128
    else:
        monkeypatch.setenv("RSB_WGRAD_DETERMINISTIC", "1")
        C, B, H, W = (2, 2, 64, 64) if cfg == "a" else (2, 2, 128, 128)
        lists = ("fwd", "bwd") if cfg == "a" else ("fwd",)
    gpu, cpu, x, dlogits = _make_engines(C, B, H, W, cuda_device)
    gpu.use_graph = False
    table = {}
    n, failures = replay_step(gpu, cpu, x, dlogits, lambda op, xg, dlg: gpu._run([op], x=xg, dlogits=dlg), torch.cuda.synchronize, table, lists)
    _print_table("config %s (%d classes, batch %d, %dx%d), %d ops" % (cfg, C, B, H, W, n), table)
    assert not failures, "\n".join(failures[:20])
    assert n == sum(len(getattr(gpu, p + "_ops")) for p in lists)
    if cfg == "c":
        assert max(-(-u.stats_rows // 32) for u in gpu.units.values() if u.stats is not None and u.desc.Cout == 64) >= 8
        return
    assert n > 400
    if cfg == "a":
        assert getattr(gpu, "_wgrad_scratch", None) is not None, "no wgrad plan used the deterministic reduce"
        assert any(item[0] == "gather" for item in gpu._unpack_all)
    else:
        assert getattr(gpu, "_wgrad_scratch", None) is None and all(item[0] == "scatter" for item in gpu._unpack_all)
