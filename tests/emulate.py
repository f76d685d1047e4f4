"""CPU emulation of the semantics of `rsb_conv_run` for descriptors whose pointers are HOST memory.

Test infrastructure only. It reads the raw pointers of an `rsb_conv_desc` exactly the way the kernel's TMA
boxes do (views with arbitrary -- possibly overlapping -- pitches, zero fill outside the view extents) so the
host-side logic (weight packing, parity views, upsample phases, window views, output addressing) can be
verified without a GPU.
"""

import ctypes

import numpy as np


def _view(ptr, shape, strides_elems, dtype=np.float16, writable=False):
    item = np.dtype(dtype).itemsize
    span = 1 + sum((s - 1) * abs(st) for s, st in zip(shape, strides_elems))
    raw = (ctypes.c_uint8 * (span * item)).from_address(ptr)
    base = np.frombuffer(raw, dtype=dtype)
    v = np.lib.stride_tricks.as_strided(base, shape=shape, strides=[st * item for st in strides_elems], writeable=writable)
    return v


def prepass_s2d_cpu(x):
    """torch fp32 NCHW -> fp16 [N, H/2, W/2+4, 16] (what rsb_prepass_s2d writes)"""
    import torch

    N, C, H, W = x.shape
    out = torch.zeros(N, H // 2, W // 2 + 4, 16, dtype=torch.float16)
    for ph in range(2):
        for pw in range(2):
            out[:, :, 2:2 + W // 2, (ph * 2 + pw) * 3:(ph * 2 + pw) * 3 + 3] = x[:, :, ph::2, pw::2].permute(0, 2, 3, 1).half()
    return out


def prepass_s2d_split_cpu(x):
    """rsb_prepass_s2d_split: [2, N, H/2, W/2+4, 16], plane 0 = half(x), plane 1 = half(x - float(half(x)))"""
    import torch

    hi = prepass_s2d_cpu(x)
    N, C, H, W = x.shape
    xs = torch.zeros(N, H // 2, W // 2 + 4, 16, dtype=torch.float32)
    for ph in range(2):
        for pw in range(2):
            xs[:, :, 2:2 + W // 2, (ph * 2 + pw) * 3:(ph * 2 + pw) * 3 + 3] = x[:, :, ph::2, pw::2].permute(0, 2, 3, 1)
    return torch.stack([hi, (xs - hi.float()).half()])


def split_pair(v32):
    """fp32 array -> (hi, lo) fp16 arrays the way the kernels' epilogues do it (residue exact in fp32)"""
    hi = v32.astype(np.float16)
    lo = (v32 - hi.astype(np.float32)).astype(np.float16)
    return hi, lo


def _pair(ptr, plane, shape, strides):
    """value of an operand view: fast mode = the fp16 plane; split mode = hi + lo (exact in fp32), as float64"""
    v = _view(ptr, shape, strides).astype(np.float64)
    if plane:
        v = v + _view(ptr + 2 * plane, shape, strides).astype(np.float64)
    return v


def run_desc(d):
    """Execute descriptor `d` (host pointers) and write its outputs like the device kernel would.
    Split descriptors: operands are hi + lo pairs; the contraction is done in float64 (the kernel's fp32 accumulation of
    hi*hi + hi*lo + lo*hi differs from it by ~1e-7 relative), the epilogue in fp32 exactly like the kernel."""
    split = bool(d.split)
    K = 64 * sum(d.segs[i].cblocks for i in range(d.nseg))
    rows = d.phases * d.Cout
    wts = _pair(d.weights, rows * K if split else 0, (rows, K), (K, 1))
    if not split:
        wts = wts.astype(np.float32)
    scale = np.float32(d.acc_scale if d.acc_scale != 0 else 1.0)
    bias = _view(d.bias, (d.Cout,), (1,), np.float32) if d.bias else None
    Nt, Ht, Wt = d.Nt, d.Ht, d.Wt
    hh0 = np.arange(Ht)[:, None]
    ww0 = np.arange(Wt)[None, :]
    acc_t = np.float64 if split else np.float32
    for phase in range(d.phases):
        pa, pb = phase >> 1, phase & 1
        acc = np.zeros((Nt, Ht, Wt, d.Cout), dtype=acc_t)
        k0 = 0
        for si in range(d.nseg):
            seg = d.segs[si]
            src = d.srcs[seg.src]
            width = seg.cblocks * 64
            sv = _pair(src.ptr, src.plane if split else 0, (src.N, src.H, src.W, min(width, src.C)), (src.pitch_n, src.pitch_h, src.pitch_w, 1))
            hh = hh0 + seg.dh + pa
            ww = ww0 + seg.dw + pb
            inb = (hh >= 0) & (hh < src.H) & (ww >= 0) & (ww < src.W)
            a = np.zeros((Nt, Ht, Wt, width), dtype=acc_t)
            g = sv[:, np.clip(hh, 0, src.H - 1), np.clip(ww, 0, src.W - 1), :].astype(acc_t)  # [N, Ht, Wt, c]
            g = g * inb[None, :, :, None]
            nn = min(Nt, src.N)
            a[:nn, :, :, :g.shape[-1]] = g[:nn]
            wseg = wts[phase * d.Cout:(phase + 1) * d.Cout, k0:k0 + width]
            acc += np.tensordot(a, wseg, axes=([3], [1]))
            k0 += width
        acc = acc.astype(np.float32) * scale
        if bias is not None:
            acc += bias
        if d.mode == 0:
            base = d.out + 2 * (pa * d.out_pitch_h + pb * d.out_pitch_w)
            strides = (d.out_pitch_n, d.out_sy * d.out_pitch_h, d.out_sx * d.out_pitch_w, 1)
            if d.residual:
                rbase = d.residual + 2 * (pa * d.out_pitch_h + pb * d.out_pitch_w)
                acc += _pair(rbase, d.res_plane if split else 0, (Nt, Ht, Wt, d.Cout), strides).astype(np.float32)
            if d.relu:
                acc = np.maximum(acc, 0)
            ov = _view(base, (Nt, Ht, Wt, d.Cout), strides, writable=True)
            if split:
                hi, lo = split_pair(acc)
                ov[...] = hi
                _view(base + 2 * d.out_plane, (Nt, Ht, Wt, d.Cout), strides, writable=True)[...] = lo
            else:
                ov[...] = acc.astype(np.float16)
        else:
            if d.relu:
                acc = np.maximum(acc, 0)
            hw = _view(d.head_w, (d.head_classes, 32), (32, 1), np.float32)
            hb = _view(d.head_b, (d.head_classes,), (1,), np.float32)
            logits = np.tensordot(acc, hw, axes=([3], [1])) + hb  # [N, H, W, classes]
            ov = _view(d.head_out, (Nt, d.head_classes, Ht, Wt), (d.head_classes * Ht * Wt, Ht * Wt, Wt, 1), np.float32, writable=True)
            ov[...] = np.transpose(logits, (0, 3, 1, 2))


def run_rowdesc(d):
    """CPU semantics of rsb_rowconv_run (line-buffer kernel): same arithmetic as run_desc, described by taps instead of segments"""
    nph = d.nphase_a * d.nsub
    K = d.taps_h * d.taps_w * d.cin
    split = bool(getattr(d, "split", 0))
    wts = _pair(d.weights, nph * d.Cout * K if split else 0, (nph * d.Cout, K), (K, 1))
    if not split:
        wts = wts.astype(np.float32)
    scale = np.float32(d.acc_scale if split and d.acc_scale != 0 else 1.0)
    bias = _view(d.bias, (d.Cout,), (1,), np.float32) if d.bias else None
    src = d.src
    sv = _pair(src.ptr, src.plane if split else 0, (src.N, src.H, src.W, d.cin), (src.pitch_n, src.pitch_h, src.pitch_w, 1))
    if not split:
        sv = sv.astype(np.float32)
    for a in range(d.nphase_a):
        for s_ in range(d.nsub):
            acc = np.zeros((d.Nt, d.Ht, d.Wt, d.Cout), dtype=np.float64 if split else np.float32)
            for th in range(d.taps_h):
                for tw in range(d.taps_w):
                    hh = np.arange(d.Ht)[:, None] + d.dh0 + a + th
                    ww = np.arange(d.Wt)[None, :] + d.dw0 + s_ + tw
                    inb = (hh >= 0) & (hh < src.H) & (ww >= 0) & (ww < src.W)
                    g = sv[:, np.clip(hh, 0, src.H - 1), np.clip(ww, 0, src.W - 1), :] * inb[None, :, :, None]
                    k0 = (th * d.taps_w + tw) * d.cin
                    wseg = wts[(a * d.nsub + s_) * d.Cout:(a * d.nsub + s_ + 1) * d.Cout, k0:k0 + d.cin]
                    acc += np.tensordot(g[:d.Nt], wseg, axes=([3], [1]))
            acc = acc.astype(np.float32) * scale
            if bias is not None:
                acc += bias
            if d.relu:
                acc = np.maximum(acc, 0)
            if d.mode == 0:
                base = d.out + 2 * (a * d.out_pitch_h + s_ * d.out_pitch_w)
                ov = _view(base, (d.Nt, d.Ht, d.Wt, d.Cout), (d.out_pitch_n, d.out_sy * d.out_pitch_h, d.out_sx * d.out_pitch_w, 1), writable=True)
                ov[...] = acc.astype(np.float16)
            else:
                hw = _view(d.head_w, (d.head_classes, 32), (32, 1), np.float32)
                hb = _view(d.head_b, (d.head_classes,), (1,), np.float32)
                logits = np.tensordot(acc, hw, axes=([3], [1])) + hb
                ov = _view(d.head_out, (d.Nt, d.head_classes, d.Ht, d.Wt), (d.head_classes * d.Ht * d.Wt, d.Ht * d.Wt, d.Wt, 1), np.float32, writable=True)
                ov[...] = np.transpose(logits, (0, 3, 1, 2))


def run_engine(engine, x):
    """Execute a plan_only UNetEngine (CPU buffers) op by op; returns fp32 NCHW logits (torch)."""
    import torch
    import torch.nn.functional as F

    assert engine.plan_only and engine.device.type == "cpu"
    strict = getattr(engine, "strict", False)
    for op in engine.ops:
        if op[0] == "prepass":
            engine.s2d.copy_(prepass_s2d_split_cpu(x) if strict else prepass_s2d_cpu(x))
        elif op[0] == "maxpool":
            _, src, dst, n, h, w, c, k, s, p = op
            if strict:
                v = (src[0].float() + src[1].float()).reshape(n, h, w, c).permute(0, 3, 1, 2)
                y = F.max_pool2d(v, kernel_size=k, stride=s, padding=p).permute(0, 2, 3, 1)
                hi = y.half()
                dst.copy_(torch.stack([hi, (y - hi.float()).half()]).reshape(dst.shape))
            else:
                y = F.max_pool2d(src.float().reshape(n, h, w, c).permute(0, 3, 1, 2), kernel_size=k, stride=s, padding=p)
                dst.copy_(y.permute(0, 2, 3, 1).half())
        elif hasattr(op[1].desc, "taps_h"):
            run_rowdesc(op[1].desc)
        else:
            run_desc(op[1].desc)
    return engine.logits.clone()


# --------------------------------------------------------------------------------------------------
# training plan emulation (robosat_b200/train_engine.py op lists on CPU buffers)
# --------------------------------------------------------------------------------------------------
def _gather_segment(d, seg, phase):
    """A operand of one segment for all tile-space pixels: float32 [Nt, Ht, Wt, 64*cblocks] (zero outside the view)"""
    pa, pb = phase >> 1, phase & 1
    src = d.srcs[seg.src]
    width = seg.cblocks * 64
    sv = _view(src.ptr, (src.N, src.H, src.W, min(width, src.C)), (src.pitch_n, src.pitch_h, src.pitch_w, 1))
    hh = np.arange(d.Ht)[:, None] + seg.dh + pa
    ww = np.arange(d.Wt)[None, :] + seg.dw + pb
    inb = (hh >= 0) & (hh < src.H) & (ww >= 0) & (ww < src.W)
    g = sv[:, np.clip(hh, 0, src.H - 1), np.clip(ww, 0, src.W - 1), :].astype(np.float32) * inb[None, :, :, None]
    a = np.zeros((d.Nt, d.Ht, d.Wt, width), dtype=np.float32)
    nn = min(d.Nt, src.N)
    a[:nn, :, :, :g.shape[-1]] = g[:nn]
    return a


def run_wgrad(d, dy_ptr, dw):
    """dw[phase*Cout + co][k] = sum_pixels dy_phase[p][co] * A_segment(k)[p]  (what rsb_wgrad_run accumulates); dw: torch fp32"""
    K = 64 * sum(d.segs[i].cblocks for i in range(d.nseg))
    out = dw.numpy().reshape(d.phases * d.Cout, K)
    out[...] = 0
    for phase in range(d.phases):
        pa, pb = phase >> 1, phase & 1
        base = dy_ptr + 2 * (pa * d.out_pitch_h + pb * d.out_pitch_w)
        dyv = _view(base, (d.Nt, d.Ht, d.Wt, d.Cout), (d.out_pitch_n, d.out_sy * d.out_pitch_h, d.out_sx * d.out_pitch_w, 1)).astype(np.float32)
        k0 = 0
        for si in range(d.nseg):
            a = _gather_segment(d, d.segs[si], phase)
            out[phase * d.Cout:(phase + 1) * d.Cout, k0:k0 + a.shape[-1]] = np.tensordot(dyv, a, axes=([0, 1, 2], [0, 1, 2]))
            k0 += a.shape[-1]


def run_train_ops(eng, ops, x=None, dlogits=None):
    """Replay a UNetTrainEngine op list (plan_only, CPU buffers) with torch / numpy semantics of the C ABI entry points."""
    import torch
    import torch.nn.functional as F

    P = eng.params
    for op in ops:
        k = op[0]
        if k == "conv":
            run_desc(op[1].desc)
        elif k == "pack_all":
            for wname, m, dst, _c, _o in eng.pack_list:
                src = P[wname].reshape(-1)
                mm = m.long()
                vals = torch.where(mm >= 0, src[mm.clamp_min(0)], torch.zeros(()))
                dst.copy_(vals.sum(1).half())
        elif k == "unpack_all":
            for dwp, m, wname, _c, _o in eng.unpack_list:
                flat = eng._grad(wname).reshape(-1)
                mm = m.long()
                for j in range(4):
                    sel = mm[:, j] >= 0
                    flat.index_add_(0, mm[sel, j], dwp[sel] / eng.loss_scale)
        elif k == "bn_stats":
            b = op[1]
            z = b.z.reshape(b.M, b.C).double()
            b.sums[:b.C] = z.sum(0)
            b.sums[b.C:2 * b.C] = (z * z).sum(0)
        elif k == "bn_finalize":
            b = op[1]
            pf = b.prefix
            mean = b.sums[:b.C] / b.M
            var = (b.sums[b.C:2 * b.C] / b.M - mean * mean).clamp_min(0)
            invstd = (1.0 / torch.sqrt(var + eng_eps())).float()
            b.mean.copy_(mean.float())
            b.invstd.copy_(invstd)
            b.scale.copy_(P[pf + ".weight"] * invstd)
            b.shift.copy_(P[pf + ".bias"] - mean.float() * b.scale)
            P[pf + ".running_mean"].mul_(0.9).add_(0.1 * mean.float())
            P[pf + ".running_var"].mul_(0.9).add_(0.1 * (var * b.M / (b.M - 1)).float())
            P[pf + ".num_batches_tracked"].add_(1)
        elif k == "bn_apply":
            _, b, res, y, relu = op
            o = b.z.reshape(b.M, b.C).float() * b.scale + b.shift
            if res is not None:
                o = o + res.reshape(b.M, b.C).float()
            y.copy_((F.relu(o) if relu else o).half().reshape(y.shape))
        elif k == "bn_bwd":
            _, b, dy, y, dz, g_out = op
            pf = b.prefix
            g = dy.reshape(b.M, b.C).float()
            if y is not None:  # masked entries are +0, as autograd's threshold_backward writes them
                g = torch.where(y.reshape(b.M, b.C).float() > 0, g, torch.zeros(()))
            zhat = (b.z.reshape(b.M, b.C).float() - b.mean) * b.invstd
            s0 = g.double().sum(0)
            s1 = (g * zhat).double().sum(0)
            if g_out is not None:
                g_out.copy_(g.half().reshape(g_out.shape))
            o = P[pf + ".weight"] * b.invstd * (g - (s0 / b.M).float() - zhat * (s1 / b.M).float())
            dz.copy_(o.half().reshape(dz.shape))
            eng._grad(pf + ".weight").copy_((s1 / eng.loss_scale).float())
            eng._grad(pf + ".bias").copy_((s0 / eng.loss_scale).float())
        elif k == "relu_bwd":
            _, a, b2, y, out = op
            g = a.float()
            if b2 is not None:
                g = g + b2.float()
            if y is not None:
                g = torch.where(y.float() > 0, g, torch.zeros(()))
            out.copy_(g.half())
        elif k == "maxpool":
            _, src, dst, n, h, w, c, kk, s, p = op
            yy = F.max_pool2d(src.float().reshape(n, h, w, c).permute(0, 3, 1, 2), kk, s, p)
            dst.copy_(yy.permute(0, 2, 3, 1).half())
        elif k == "maxpool_bwd":
            _, xx, dy, dx, n, h, w, c, kk, s, p = op
            xin = xx.float().reshape(n, h, w, c).permute(0, 3, 1, 2).clone().requires_grad_(True)
            yy = F.max_pool2d(xin, kk, s, p)
            yy.backward(dy.float().reshape(n, yy.shape[2], yy.shape[3], c).permute(0, 3, 1, 2))
            dx.copy_(xin.grad.permute(0, 2, 3, 1).half())
        elif k == "wgrad":
            _, u, dy = op
            run_wgrad(u.desc, dy.data_ptr() + 2 * u.out_offset, u.dw_packed)
        elif k == "prepass":
            eng.s2d.copy_(prepass_s2d_cpu(x))
        elif k == "final_fwd":
            _, y5, logits = op
            yv = y5.float().permute(0, 3, 1, 2)
            logits.copy_(F.conv2d(yv, P["final.weight"], P["final.bias"]))
        elif k == "final_bwd":
            _, y5, d_y5 = op
            w = P["final.weight"].reshape(eng.C, 32)
            d = torch.einsum("nkhw,kc->nhwc", dlogits, w) * eng.loss_scale
            d_y5.copy_(d.half())
            eng._grad("final.weight").copy_(torch.einsum("nkhw,nhwc->kc", dlogits, y5.float()).reshape(eng.C, 32, 1, 1))
            eng._grad("final.bias").copy_(dlogits.sum((0, 2, 3)))
        elif k == "zero_grads":
            eng._grad("final.bias")
            eng._grads_flat.zero_()
        else:
            raise AssertionError(k)


def eng_eps():
    return 1e-5


def stitch_halo_cpu(store, table, size, overlap):
    """numpy restatement of csrc/rsb_elementwise.cu:stitch_halo_kernel (same index arithmetic), for the CPU suite."""
    import numpy as np

    B = table.shape[0]
    F = size + 2 * overlap
    out = np.zeros((B, F, F, 3), dtype=np.uint8)
    for b in range(B):
        for Y in range(F):
            dy = -1 if Y < overlap else (0 if Y < overlap + size else 1)
            sy = Y - overlap - dy * size
            for dx, (x0, x1) in ((-1, (0, overlap)), (0, (overlap, overlap + size)), (1, (overlap + size, F))):
                if x1 <= x0:
                    continue
                slot = int(table[b, (dy + 1) * 3 + (dx + 1)])
                if slot < 0:
                    continue
                out[b, Y, x0:x1] = store[slot, sy, x0 - overlap - dx * size:x1 - overlap - dx * size]
    return out
