"""Host-side plan of one U-Net TRAINING step (forward in train mode + full backward) on librsb200.so.

Replaces what `outputs = net(images); loss.backward()` does in the reference's hot loop
(robosat/tools/train.py:180,186) for `UNet` (robosat/unet.py:110-141) with train-mode BatchNorm (torchvision resnet50):

  forward   per conv: fp32 master weights -> fp16 packed (rsb_pack_weights) -> tcgen05 conv (raw output z)
            -> batch statistics (rsb_bn_stats / rsb_bn_finalize, running stats updated) -> y = relu(bn(z) (+ identity))
            decoder convs have no BN: y = relu(conv) in the conv epilogue; final 1x1 conv is its own small kernel
  backward  per conv: BN / ReLU backward (rsb_bn_backward, rsb_relu_backward) -> weight gradient on tensor cores in the
            forward's packed layout (rsb_wgrad_*) -> rsb_unpack_grads to OIHW fp32 -> input gradient = the SAME conv
            kernel with transposed / flipped packed weights (strided convs and the fused upsample become 4-phase scatters,
            concat becomes one launch per source, fan-in sums ride on the kernel's residual input)

The engine only builds buffers, descriptors and two op lists (`fwd_ops`, `bwd_ops`); an executor replays them. The GPU
executor calls the C ABI; tests/emulate.py replays the same lists on the CPU to check the host logic against autograd.
Activation gradients are fp16 and carry `loss_scale`; parameter gradients are fp32 and unscaled.

precision="strict" (opt-in; RSB_TRAIN_PRECISION) keeps every forward activation as an fp16 (hi, lo) pair, like the strict inference
plan: split convolutions, BatchNorm statistics of hi + lo in fp64, BN apply / max pool / final 1x1 on the fp32 values hi + lo. The
backward is the fast one on the hi planes, with every ReLU mask and max-pool arg-max taken from what the strict forward applied.
"""

import ctypes
import math
import os
from collections import OrderedDict

import numpy as np
import torch

from robosat_b200 import _lib
from robosat_b200._lib import ConvDesc, ConvSrc

# BatchNorm kernels chained by programmatic dependent launch, accumulators cleaned by the kernels themselves (no memset launches)
TRAIN_GRAPH = os.environ.get("RSB_TRAIN_GRAPH", "1") == "1"  # forward / backward op lists replayed from CUDA graphs
CONV_STATS = os.environ.get("RSB_CONV_STATS", "1") == "1"  # BatchNorm batch sums from the conv epilogue (profiles/r2_train.md)
BN_CHAINED = os.environ.get("RSB_BN_CHAINED", "1") == "1"  # measured: 17.77 vs 18.03 ms per cfg-3 step (profiles/r2_train.md)
from robosat_b200.engine import ConvOp, _src_dense, _src_parity, make_conv_desc

TRAIN_PRECISIONS = ("fast", "strict")
# strict plans scale every forward weight layout by a power of two fixed when the plan is built: its largest |w| lands in
# [2^9, 2^10), so the weights may grow 64x before a scaled hi overflows fp16 (counted on the device; the owner rebuilds the plan)
STRICT_WEIGHT_EXP = 9


def default_train_precision():
    """`fast` (single fp16 forward activations) unless RSB_TRAIN_PRECISION=strict (hi/lo fp16 pairs: fp32-class forward)"""
    p = os.environ.get("RSB_TRAIN_PRECISION", "fast").lower()
    if p not in TRAIN_PRECISIONS:
        raise ValueError("RSB_TRAIN_PRECISION must be one of %s" % (TRAIN_PRECISIONS,))
    return p

RESNET50_BLOCKS = (3, 4, 6, 3)
BN_EPS = 1e-5
BN_MOMENTUM = 0.1
_UP_GROUPS = {0: ((0,), (1, 2)), 1: ((0, 1), (2,))}  # rows of the 3x3 kernel summed per (phase a, tap th)


# --------------------------------------------------------------------------------------------------
# index maps: packed element -> up to 4 flat OIHW source indices (-1 = none). One map drives rsb_pack_weights
# (gather + sum) and, for forward layouts, rsb_unpack_grads (scatter-add).
# --------------------------------------------------------------------------------------------------
def _flat_index(shape):
    return np.arange(int(np.prod(shape)), dtype=np.int64).reshape(shape)


def _map4(single):
    """[...] int64 gather map (with -1) -> [n, 4] int32"""
    m = np.full((single.size, 4), -1, dtype=np.int32)
    m[:, 0] = single.reshape(-1)
    return m


def map_conv_fwd(shape):
    idx = _flat_index(shape)  # [co, ci, kh, kw]
    return _map4(idx.transpose(0, 2, 3, 1))  # [co][kh][kw][ci]


def map_conv_dgrad(shape, pad_co_to=None):
    """stride-1 dgrad operand: rows = ci, K = (kh', kw', co) with the taps flipped; co optionally zero-padded to a 64-block"""
    co, ci, kh, kw = shape
    idx = _flat_index(shape)[:, :, ::-1, ::-1].transpose(1, 2, 3, 0)  # [ci][kh'][kw'][co]
    if pad_co_to and pad_co_to > co:
        full = np.full((ci, kh, kw, pad_co_to), -1, dtype=np.int64)
        full[..., :co] = idx
        idx = full
    return _map4(idx)


def map_up_fwd(shape):
    """fused nearest-x2 + 3x3: [phase][co][(th,tw)][ci] <- sum of the taps of group (a,th) x (b,tw)"""
    co, ci, _, _ = shape
    idx = _flat_index(shape)
    m = np.full((4, co, 2, 2, ci, 4), -1, dtype=np.int32)
    for a in (0, 1):
        for b in (0, 1):
            for th in (0, 1):
                for tw in (0, 1):
                    j = 0
                    for kh in _UP_GROUPS[a][th]:
                        for kw in _UP_GROUPS[b][tw]:
                            m[2 * a + b, :, th, tw, :, j] = idx[:, :, kh, kw]
                            j += 1
    return m.reshape(-1, 4)


def map_up_dgrad(shape, ci_lo, ci_hi, pad_co_to):
    """dgrad of the fused upsample conv w.r.t. source channels [ci_lo, ci_hi): rows = ci, K = 16 segments
    (a, b, th, tw) x co (padded to a 64-block), each the transposed phase weight block (sum of its taps)."""
    co, _, _, _ = shape
    idx = _flat_index(shape)
    n_ci = ci_hi - ci_lo
    m = np.full((n_ci, 2, 2, 2, 2, pad_co_to, 4), -1, dtype=np.int32)
    for a in (0, 1):
        for b in (0, 1):
            for th in (0, 1):
                for tw in (0, 1):
                    j = 0
                    for kh in _UP_GROUPS[a][th]:
                        for kw in _UP_GROUPS[b][tw]:
                            m[:, a, b, th, tw, :co, j] = idx[:, ci_lo:ci_hi, kh, kw].T
                            j += 1
    return m.reshape(-1, 4)


def map_s2_dgrad(shape):
    """dgrad of a 3x3 stride-2 pad-1 conv as 4 output phases of 2x2 taps on dy: [phase][ci][(th,tw)][co]"""
    co, ci, _, _ = shape
    idx = _flat_index(shape)
    ksel = {(0, 0): None, (0, 1): 1, (1, 0): 2, (1, 1): 0}  # (phase bit, tap) -> kernel index
    m = np.full((4, ci, 2, 2, co), -1, dtype=np.int64)
    for a in (0, 1):
        for b in (0, 1):
            for th in (0, 1):
                for tw in (0, 1):
                    kh, kw = ksel[(a, th)], ksel[(b, tw)]
                    if kh is None or kw is None:
                        continue
                    m[2 * a + b, :, th, tw, :] = idx[:, :, kh, kw].T
    return _map4(m)


def map_stem_fwd(shape):
    co = shape[0]
    idx = _flat_index(shape)
    m = np.full((co, 4, 4, 16), -1, dtype=np.int64)
    for t in range(4):
        for ph in range(2):
            kh = 2 * t + ph - 1
            if not 0 <= kh < 7:
                continue
            for u in range(4):
                for pw in range(2):
                    kw = 2 * u + pw - 1
                    if not 0 <= kw < 7:
                        continue
                    m[:, t, u, (ph * 2 + pw) * 3:(ph * 2 + pw) * 3 + 3] = idx[:, :, kh, kw]
    return _map4(m)


def map_window3_fwd(shape):
    co, ci, _, _ = shape
    idx = _flat_index(shape)
    m = np.full((co, 3, 4, ci), -1, dtype=np.int64)
    m[:, :, :3, :] = idx.transpose(0, 2, 3, 1)
    return _map4(m)


class Unit:
    """One convolution of the network with everything its forward and backward need."""

    def __init__(self, name):
        self.name = name


class UNetTrainEngine:
    def __init__(self, params, num_classes, batch, height, width, device="cuda", loss_scale=4096.0, plan_only=False, precision=None):
        """params: name -> fp32 tensor on `device` with the reference's state_dict names WITHOUT the `module.` prefix
        (weights, BN affine + running stats + num_batches_tracked). They are read (and the BN buffers updated) in place.
        Gradients are written to `self.grads[name]` (fp32, zeroed at the start of every backward).

        precision: "fast" (single fp16 forward activations and weights), "strict" (every forward activation an fp16 (hi, lo) pair,
        split convolutions with three MMAs per K step, BatchNorm statistics in fp64 from hi + lo: train-mode logits, batch
        statistics, ReLU masks and max-pool arg-maxes at fp32 level; the backward is the fast one, reading the hi planes) or None
        (RSB_TRAIN_PRECISION, default fast)."""
        assert height % 64 == 0 and width % 64 == 0
        self.precision = default_train_precision() if precision is None else precision
        if self.precision not in TRAIN_PRECISIONS:
            raise ValueError("precision must be one of %s, not %r" % (TRAIN_PRECISIONS, precision))
        self.strict = self.precision == "strict"
        self.plan_only = plan_only
        if not plan_only:
            _lib.require_device()
        self.device = torch.device(device)
        self.N, self.H, self.W, self.C = batch, height, width, num_classes
        self.params = params
        self.loss_scale = float(loss_scale)
        self.fwd_ops, self.bwd_ops = [], []
        self.pack_list, self.unpack_list = [], []  # (wname, map, packed fp16) / (packed fp32 grad, map, wname)
        self._pack_all = None
        self._stats_buf = {}
        self._graphs = {}
        self.use_graph = TRAIN_GRAPH and not plan_only
        self._pack_chunks = []  # [fp16 arena tensor, elements used]
        self._dw_chunks = []    # [fp32 arena tensor, elements used] packed weight gradients
        self._grads_flat, self._grad_offset, self._unpack_all = None, {}, None
        self._keep = []
        self._pool_scratch = {}  # max-pool backward: one argmax byte per pooled element
        self._accum_tables = {}
        self.grads = OrderedDict()
        self.units = OrderedDict()
        self.feats = OrderedDict()
        self.relu_outs = OrderedDict()  # name -> (post-ReLU activation buffer, logical NHWC shape): masks for tests / debugging
        # strict: forward weight layouts packed as (hi, lo) planes of w * 2^e, one exponent per layout; weights past it are counted
        self.split_pack_list = []  # (wname, map, packed fp16 [2][n], 2^e, one source per element?)
        self.exponents = OrderedDict()  # unit name -> e (the unit's forward descriptor has acc_scale = 2^-e)
        self._pair_planes = {}  # data_ptr -> plane stride of every two-plane forward activation buffer
        self.overflow = self._buf(1, dtype=torch.int32) if self.strict else None
        self._overflow_host, self._overflow_event = None, None
        self._build()

    # ---------------------------------------------------------------- allocation helpers
    def _buf(self, *shape, dtype=torch.float16):
        t = torch.zeros(shape, dtype=dtype, device=self.device)
        self._keep.append(t)
        return t

    def _dev(self, arr, dtype=None):
        t = torch.as_tensor(arr)
        if dtype is not None:
            t = t.to(dtype)
        t = t.contiguous().to(self.device)
        self._keep.append(t)
        return t

    def _grad(self, name):
        """fp32 gradient of parameter `name`: a view of ONE flat buffer (zeroed with a single memset per backward)"""
        if self._grads_flat is None:
            names = [k for k, v in self.params.items()
                     if v.dtype == torch.float32 and not k.endswith("running_mean") and not k.endswith("running_var") and not k.startswith("resnet.fc.")]
            total = sum(self.params[k].numel() for k in names)
            self._grads_flat = torch.zeros(total, dtype=torch.float32, device=self.device)
            off = 0
            for k in names:
                n = self.params[k].numel()
                self.grads[k] = self._grads_flat[off:off + n].view(tuple(self.params[k].shape))
                self._grad_offset[k] = off
                off += n
        return self.grads[name]

    def _act(self, *shape):
        """forward activation buffer: NHWC fp16, with a leading (hi, lo) plane axis in strict precision"""
        if not self.strict:
            return self._buf(*shape)
        t = self._buf(2, *shape)
        self._pair_planes[t.data_ptr()] = t.numel() // 2
        return t

    def _plane(self, t):
        return self._pair_planes.get(t.data_ptr(), 0) if t is not None else 0

    def _hi(self, t):
        """the single fp16 view the backward kernels read: the hi plane of a two-plane activation (the buffer itself otherwise)"""
        return t[0] if self._plane(t) else t

    def _dense(self, t, N, H, W, C):
        return _src_dense(t, N, H, W, C, self._plane(t))

    def _parity(self, t, N, H, W, C, ph, pw):
        return _src_parity(t, N, H, W, C, ph, pw, self._plane(t))

    def _scratch(self):
        """one fp32 scratch tile per SM for the K-chunked split convolutions, shared by all layers (launches are stream ordered)"""
        if getattr(self, "_scratch_buf", None) is None:
            n = 148 * 128 * 256 if self.plan_only else int(_lib.load().rsb_conv_scratch_bytes(256)) // 4
            self._scratch_buf = self._buf(n, dtype=torch.float32)
        return self._scratch_buf

    def _packed_split(self, name, wname, m):
        """strict forward layout of `wname` (m: device map [n, 4]): fp16 [2][n] (hi, lo) of the packed weights times 2^e, refreshed
        by pack_all every step. e is fixed here from the current weights (it is baked into the conv's acc_scale and the captured
        graphs)."""
        src = self.params[wname].detach().reshape(-1)
        mm = m.long()
        vals = torch.where(mm >= 0, src[mm.clamp_min(0)], torch.zeros((), device=src.device)).sum(1)
        amax = float(vals.abs().max())
        e = STRICT_WEIGHT_EXP - int(math.floor(math.log2(amax))) if math.isfinite(amax) and amax > 0 else 0
        single = bool((m[:, 1:] < 0).all())
        dm = self._dev(m[:, 0], torch.int32) if single else m
        dst = self._buf(2, m.shape[0])
        self.split_pack_list.append((wname, dm, dst, 2.0 ** e, single))
        self.exponents[name] = e
        return dst, 2.0 ** -e

    def _conv_op(self, name, desc):
        return ConvOp(name, desc, (), create_plan=not self.plan_only)

    def _packed(self, wname, map4):
        """(packed fp16 buffer, device map) for parameter `wname`; refreshed from the fp32 master weights once per step
        by the ("pack_all",) op at the head of the forward program (one launch for every operand layout of every layer when
        the parameters live in one arena, e.g. robosat_b200.optim.Adam's)"""
        m = self._dev(map4, torch.int32)
        n = m.shape[0]
        # bump-allocate the packed buffer inside a shared fp16 arena chunk (16-byte aligned for TMA)
        chunk_elems = 48 * 1024 * 1024
        if not self._pack_chunks or self._pack_chunks[-1][1] + n > self._pack_chunks[-1][0].numel():
            self._pack_chunks.append([self._buf(max(chunk_elems, n)), 0])
        chunk, used = self._pack_chunks[-1]
        dst = chunk[used:used + n]
        self._pack_chunks[-1][1] = used + ((n + 7) // 8) * 8
        self.pack_list.append((wname, m, dst, len(self._pack_chunks) - 1, used))
        return dst, m

    # ---------------------------------------------------------------- unit construction
    def _add_unit(self, name, wname, fwd_map, srcs, segs, cout, phases, tile_space, out, out_pitches, out_scale=(1, 1), relu=False,
                  out_offset=0, residual=None, stats=False, stats_slot=0):
        """forward conv (raw output unless relu=True) + its weight-gradient plan. stats=True (a conv feeding BatchNorm): the
        epilogue also writes the per-quarter-tile column sums / sums of squares that rsb_bn_partials_finalize folds, so the
        batch statistics do not re-read z (RSB_CONV_STATS=0 keeps the separate reduction over z)."""
        u = Unit(name)
        u.wname = wname
        w = self.params[wname]
        u.wshape = tuple(w.shape)
        K = 64 * sum(s[3] for s in segs)
        if self.strict:
            # split forward (raw z, or ReLU in the epilogue); the weight gradient runs on a single-plane copy of the descriptor
            # (hi planes of the sources, which are the buffer bases)
            u.fwd_map = self._dev(fwd_map, torch.int32)
            u.w_packed, acc_scale = self._packed_split(name, wname, u.fwd_map)
            u.desc = make_conv_desc(srcs, segs, u.w_packed.view(2, phases * cout, K), None, cout, phases, tile_space, out, out_pitches,
                                    out_scale=out_scale, relu=relu, out_offset_elems=out_offset, residual=residual, split=True,
                                    acc_scale=acc_scale, out_plane=self._plane(out), res_plane=self._plane(residual), scratch=self._scratch())
            u.wdesc = ConvDesc.from_buffer_copy(u.desc)
            wd = u.wdesc
            wd.split, wd.acc_scale, wd.out_plane, wd.res_plane, wd.kchunk, wd.scratch, wd.scratch_bytes = 0, 1.0, 0, 0, 0, None, 0
            for i in range(wd.nsrc):
                wd.srcs[i].plane = 0
            stats = False  # conv-epilogue statistics are single-plane only: the strict plan reduces hi + lo in rsb_bn_stats_finalize_split
        else:
            u.w_packed, u.fwd_map = self._packed(wname, fwd_map)
            wp = u.w_packed.view(phases * cout, K)
            u.desc = make_conv_desc(srcs, segs, wp, None, cout, phases, tile_space, out, out_pitches, out_scale=out_scale, relu=relu,
                                    out_offset_elems=out_offset, residual=residual)
            u.wdesc = u.desc
        u.stats, u.stats_rows = None, 0
        if stats and CONV_STATS:
            d = u.desc
            rows = 4 * (-(-d.Wt // d.TW)) * (-(-d.Ht // d.TH)) * (-(-d.Nt // d.TN))
            need = rows * 2 * cout
            # one buffer per slot for every layer (stream ordered: written by the conv, folded before the next conv of the same slot
            # runs), grown if a later layer is larger. Slot 1: the downsample conv, which runs between conv3 and bn3's statistics.
            if self._stats_buf.get(stats_slot) is None or self._stats_buf[stats_slot].numel() < need:
                self._stats_buf[stats_slot] = self._buf(need, dtype=torch.float32)
            u.stats, u.stats_rows = self._stats_buf[stats_slot], rows
            d.stats = u.stats.data_ptr()
            d.stats_bytes = u.stats.numel() * 4
        u.fwd = self._conv_op(name, u.desc)
        nd = phases * cout * K
        if not self._dw_chunks or self._dw_chunks[-1][1] + nd > self._dw_chunks[-1][0].numel():
            self._dw_chunks.append([self._buf(max(32 * 1024 * 1024, nd), dtype=torch.float32), 0])
        dchunk, dused = self._dw_chunks[-1]
        u.dw_packed = dchunk[dused:dused + nd]
        u.dw_chunk, u.dw_off = len(self._dw_chunks) - 1, dused
        self._dw_chunks[-1][1] = dused + ((nd + 3) // 4) * 4
        u.out, u.out_offset = out, out_offset
        self.units[name] = u
        self.fwd_ops.append(("conv", u.fwd))
        return u

    def _wgrad_scratch_for(self, plan):
        """Deterministic split-K (default; RSB_WGRAD_DETERMINISTIC=0 restores fp32 atomics): one scratch for the per-slice partial
        gradients, shared by every wgrad plan of the engine (launches are stream ordered) and grown to the largest request."""
        if os.environ.get("RSB_WGRAD_DETERMINISTIC", "1") == "0":
            return
        lib = _lib.load()
        plans = self.__dict__.setdefault("_wgrad_plans", [])
        plans.append(plan)
        need = int(lib.rsb_wgrad_plan_scratch_bytes(plan))
        buf = self.__dict__.get("_wgrad_scratch")
        if need and (buf is None or buf.numel() * 4 < need):
            buf = self._wgrad_scratch = torch.empty((need + 3) // 4, dtype=torch.float32, device=self.device)
            for pl in plans[:-1]:  # plans created earlier move to the larger buffer
                if lib.rsb_wgrad_plan_scratch_bytes(pl):
                    _lib.check(lib.rsb_wgrad_plan_set_scratch(pl, buf.data_ptr(), buf.numel() * 4), "rsb_wgrad_plan_set_scratch")
        if need:
            _lib.check(lib.rsb_wgrad_plan_set_scratch(plan, buf.data_ptr(), buf.numel() * 4), "rsb_wgrad_plan_set_scratch")

    def _wgrad_ops(self, u, dy):
        """weight gradient of unit u from dy (addressed like u's forward output), unpacked into the OIHW gradient"""
        self._grad(u.wname)
        self.unpack_list.append((u.dw_packed, u.fwd_map, u.wname, u.dw_chunk, u.dw_off))
        return [("wgrad", u, dy)]

    def _dgrad(self, name, wname, map4, srcs, segs, cout, phases, tile_space, out, out_pitches, out_scale=(1, 1), residual=None,
               out_offset=0):
        """input-gradient conv: same kernel, weights re-packed by `map4` every step"""
        wp, m = self._packed(wname, map4)
        K = 64 * sum(s[3] for s in segs)
        desc = make_conv_desc(srcs, segs, wp.view(phases * cout, K), None, cout, phases, tile_space, out, out_pitches, out_scale=out_scale,
                              relu=False, residual=residual, out_offset_elems=out_offset)
        op = self._conv_op(name, desc)
        return [("conv", op)]

    def _bn(self, prefix, z, M, C, conv=None):
        b = Unit(prefix)
        # b.z: what the backward reads (the hi plane in strict precision); b.zpair / b.zplane: the two-plane forward value
        b.prefix, b.z, b.M, b.C = prefix, self._hi(z), M, C
        b.zpair, b.zplane = z, self._plane(z)
        b.partials, b.partial_rows = (conv.stats, conv.stats_rows) if conv is not None and conv.stats is not None else (None, 0)
        b.sums = self._buf(20 * C, dtype=torch.float64)  # 8 accumulator slots x {sum0, sum1} x C, arrival counter, backward coefficients
        b.mean, b.invstd, b.scale, b.shift = (self._buf(C, dtype=torch.float32) for _ in range(4))
        return b

    def _bn_fwd_ops(self, b, y, residual, relu):
        if self.strict:
            # statistics of hi + lo (fp64), apply in fp32 to a (hi, lo) pair. The backward masks by y (hi plane), never by a mask
            # re-derived from single-plane z
            self.fwd_ops.append(("bn_stats_split", b))
            self.fwd_ops.append(("bn_apply_split", b, residual, y, relu))
            b.plain_relu_y = None
            return
        self.fwd_ops.append(("bn_stats", b))
        self.fwd_ops.append(("bn_finalize", b))
        self.fwd_ops.append(("bn_apply", b, residual, y, relu))
        b.plain_relu_y = y if (residual is None and relu) else None

    # ---------------------------------------------------------------- graph
    def _build(self):
        P = self.params
        N, H, W = self.N, self.H, self.W
        H2, W2, H4, W4 = H // 2, W // 2, H // 4, W // 4
        bwd = []  # built in forward order as blocks of ops; emitted reversed at the end

        def dense(h, w, c):
            return (c, w * c, h * w * c)

        # ---- stem
        self.x_in = None
        self.s2d = self._act(N, H2, W2 + 4, 16)
        self.fwd_ops.append(("pack_all",))
        self.fwd_ops.append(("prepass_split",) if self.strict else ("prepass",))
        Wp = W2 + 4
        z0 = self._act(N, H2, W2, 64)
        y0 = self._act(N, H2, W2, 64)
        src = ConvSrc(self.s2d.data_ptr(), 16, Wp * 16, H2 * Wp * 16, 64, W2, H2, N, self._plane(self.s2d))
        stem = self._add_unit("stem", "resnet.conv1.weight", map_stem_fwd(tuple(P["resnet.conv1.weight"].shape)), [src],
                              [(0, t - 2, 0, 1) for t in range(4)], 64, 1, (W2, H2, N), z0, dense(H2, W2, 64), stats=True)
        bn0 = self._bn("resnet.bn1", z0, N * H2 * W2, 64, conv=stem)
        self._bn_fwd_ops(bn0, y0, None, True)
        p0 = self._act(N, H4, W4, 64)
        self.fwd_ops.append(("maxpool_split" if self.strict else "maxpool", y0, p0, N, H2, W2, 64, 3, 2, 1))
        self.feats["stem"] = (y0, (N, H2, W2, 64))
        self.relu_outs["stem"] = (y0, (N, H2, W2, 64))
        self.feats["enc0"] = (p0, (N, H4, W4, 64))
        d_p0 = self._buf(N, H4, W4, 64)   # gradient w.r.t. p0, produced by layer1.0's backward
        d_y0 = self._buf(N, H2, W2, 64)
        dz0 = self._buf(N, H2, W2, 64)
        bwd.append([("maxpool_bwd_split" if self.strict else "maxpool_bwd", y0, d_p0, d_y0, N, H2, W2, 64, 3, 2, 1),
                    ("bn_bwd", bn0, d_y0, self._hi(y0), dz0, None)] + self._wgrad_ops(stem, dz0))

        # ---- encoder
        cur, curC, curH, curW, d_cur = p0, 64, H4, W4, d_p0
        encs = []
        for li, blocks in enumerate(RESNET50_BLOCKS, start=1):
            planes = 64 * 2 ** (li - 1)
            for bi in range(blocks):
                p = "resnet.layer%d.%d" % (li, bi)
                stride = 2 if (bi == 0 and li > 1) else 1
                oH, oW = curH // stride, curW // stride
                outC = planes * 4
                has_ds = (p + ".downsample.0.weight") in P
                M_in, M_out = N * curH * curW, N * oH * oW
                # forward
                z1, y1 = self._act(N, curH, curW, planes), self._act(N, curH, curW, planes)
                u1 = self._add_unit(p + ".conv1", p + ".conv1.weight", map_conv_fwd(tuple(P[p + ".conv1.weight"].shape)),
                                    [self._dense(cur, N, curH, curW, curC)], [(0, 0, 0, curC // 64)], planes, 1, (curW, curH, N), z1,
                                    dense(curH, curW, planes), stats=True)
                b1 = self._bn(p + ".bn1", z1, M_in, planes, conv=u1)
                self._bn_fwd_ops(b1, y1, None, True)
                z2, y2 = self._act(N, oH, oW, planes), self._act(N, oH, oW, planes)
                if stride == 1:
                    srcs2 = [self._dense(y1, N, curH, curW, planes)]
                    segs2 = [(0, kh - 1, kw - 1, planes // 64) for kh in range(3) for kw in range(3)]
                else:
                    srcs2 = [self._parity(y1, N, curH, curW, planes, ph, pw) for ph in range(2) for pw in range(2)]
                    segs2 = [(((kh - 1) % 2) * 2 + (kw - 1) % 2, (kh - 1) // 2, (kw - 1) // 2, planes // 64) for kh in range(3) for kw in range(3)]
                u2 = self._add_unit(p + ".conv2", p + ".conv2.weight", map_conv_fwd(tuple(P[p + ".conv2.weight"].shape)), srcs2, segs2,
                                    planes, 1, (oW, oH, N), z2, dense(oH, oW, planes), stats=True)
                b2 = self._bn(p + ".bn2", z2, M_out, planes, conv=u2)
                self._bn_fwd_ops(b2, y2, None, True)
                z3 = self._act(N, oH, oW, outC)
                u3 = self._add_unit(p + ".conv3", p + ".conv3.weight", map_conv_fwd(tuple(P[p + ".conv3.weight"].shape)),
                                    [self._dense(y2, N, oH, oW, planes)], [(0, 0, 0, planes // 64)], outC, 1, (oW, oH, N), z3, dense(oH, oW, outC),
                                    stats=True)
                b3 = self._bn(p + ".bn3", z3, M_out, outC, conv=u3)
                if has_ds:
                    zd, idt = self._act(N, oH, oW, outC), self._act(N, oH, oW, outC)
                    sd_ = self._dense(cur, N, curH, curW, curC) if stride == 1 else self._parity(cur, N, curH, curW, curC, 0, 0)
                    ud = self._add_unit(p + ".downsample", p + ".downsample.0.weight", map_conv_fwd(tuple(P[p + ".downsample.0.weight"].shape)),
                                        [sd_], [(0, 0, 0, curC // 64)], outC, 1, (oW, oH, N), zd, dense(oH, oW, outC),
                                        stats=True, stats_slot=1)
                    bd = self._bn(p + ".downsample.1", zd, M_out, outC, conv=ud)
                    self._bn_fwd_ops(bd, idt, None, False)
                else:
                    idt = cur
                out = self._act(N, oH, oW, outC)
                self._bn_fwd_ops(b3, out, idt, True)
                self.feats[p] = (out, (N, oH, oW, outC))
                self.relu_outs[p + ".relu1"] = (y1, (N, curH, curW, planes))
                self.relu_outs[p + ".relu2"] = (y2, (N, oH, oW, planes))
                self.relu_outs[p + ".out"] = (out, (N, oH, oW, outC))
                d_out = self._buf(N, oH, oW, outC)  # gradient w.r.t. this block's output (written by its consumers)

                # backward of this block (executed after all later blocks)
                ops = []
                dz3, g = self._buf(N, oH, oW, outC), self._buf(N, oH, oW, outC)
                ops.append(("bn_bwd", b3, d_out, self._hi(out), dz3, g))
                ops += self._wgrad_ops(u3, dz3)
                dy2 = self._buf(N, oH, oW, planes)
                ops += self._dgrad(p + ".conv3.dgrad", p + ".conv3.weight", map_conv_dgrad(u3.wshape), [_src_dense(dz3, N, oH, oW, outC)],
                                   [(0, 0, 0, outC // 64)], planes, 1, (oW, oH, N), dy2, dense(oH, oW, planes))
                dz2 = self._buf(N, oH, oW, planes)
                ops.append(("bn_bwd", b2, dy2, self._hi(y2), dz2, None))
                ops += self._wgrad_ops(u2, dz2)
                dy1 = self._buf(N, curH, curW, planes)
                if stride == 1:
                    ops += self._dgrad(p + ".conv2.dgrad", p + ".conv2.weight", map_conv_dgrad(u2.wshape), [_src_dense(dz2, N, oH, oW, planes)],
                                       [(0, kh - 1, kw - 1, planes // 64) for kh in range(3) for kw in range(3)], planes, 1, (oW, oH, N), dy1,
                                       dense(curH, curW, planes))
                else:
                    ops += self._dgrad(p + ".conv2.dgrad", p + ".conv2.weight", map_s2_dgrad(u2.wshape), [_src_dense(dz2, N, oH, oW, planes)],
                                       [(0, th - 1, tw - 1, planes // 64) for th in range(2) for tw in range(2)], planes, 4, (oW, oH, N), dy1,
                                       dense(curH, curW, planes), out_scale=(2, 2))
                dz1 = self._buf(N, curH, curW, planes)
                ops.append(("bn_bwd", b1, dy1, self._hi(y1), dz1, None))
                ops += self._wgrad_ops(u1, dz1)
                if has_ds:
                    dzd = self._buf(N, oH, oW, outC)
                    ops.append(("bn_bwd", bd, g, None, dzd, None))
                    ops += self._wgrad_ops(ud, dzd)
                    # the downsample's input gradient lands on the (even) pixels of d_cur IN PLACE, on top of whatever the
                    # decoder's skip connection already accumulated there (residual = the buffer itself)
                    # (layer1.0 has no skip gradient underneath: plain write)
                    ops += self._dgrad(p + ".downsample.dgrad", p + ".downsample.0.weight", map_conv_dgrad(ud.wshape),
                                       [_src_dense(dzd, N, oH, oW, outC)], [(0, 0, 0, outC // 64)], curC, 1, (oW, oH, N), d_cur,
                                       dense(curH, curW, curC), out_scale=(stride, stride), residual=d_cur if li > 1 else None)
                    fan_in = d_cur
                else:
                    fan_in = g
                # d_cur = conv1 input gradient + identity / downsample gradient (in place when fan_in is d_cur itself)
                ops += self._dgrad(p + ".conv1.dgrad", p + ".conv1.weight", map_conv_dgrad(u1.wshape), [_src_dense(dz1, N, curH, curW, planes)],
                                   [(0, 0, 0, planes // 64)], curC, 1, (curW, curH, N), d_cur, dense(curH, curW, curC), residual=fan_in)
                bwd.append(ops)
                cur, curC, curH, curW, d_cur = out, outC, oH, oW, d_out
            encs.append((cur, curC, curH, curW, d_cur))
            self.feats["enc%d" % li] = (cur, (N, curH, curW, curC))
        (enc1, c1, h1, w1, d_enc1), (enc2, c2, h2, w2, d_enc2), (enc3, c3, h3, w3, d_enc3), (enc4, c4, h4, w4, d_enc4) = encs
        self._skip_grads = [d_enc1, d_enc2, d_enc3, d_enc4]

        # ---- center + decoder
        hp, wpx = h4 // 2, w4 // 2
        pool4 = self._act(N, hp, wpx, c4)
        self.fwd_ops.append(("maxpool_split" if self.strict else "maxpool", enc4, pool4, N, h4, w4, c4, 2, 2, 0))
        d_pool4 = self._buf(N, hp, wpx, c4)

        dec_bwd = []

        def decoder(name, sources, lh, lw, cout, out, out_pitches, d_out, d_out_pitches, d_sources, out_offset=0, first_into=None):
            """sources: [(tensor, C)]; d_sources: [(grad tensor, accumulate?)] receiving the input gradients"""
            wname = name + ".block.block.weight"
            wshape = tuple(P[wname].shape)
            srcs = [self._dense(t, N, lh, lw, c) for t, c in sources]
            segs = [(si, th - 1, tw - 1, c // 64) for th in range(2) for tw in range(2) for si, (_, c) in enumerate(sources)]
            u = self._add_unit(name, wname, map_up_fwd(wshape), srcs, segs, cout, 4, (lw, lh, N), out, out_pitches, out_scale=(2, 2), relu=True,
                               out_offset=out_offset)
            # backward: g = d_out * (out > 0) in place over the whole buffer, wgrad, then one dgrad launch per source
            ops = [("relu_bwd", d_out, None, self._hi(out), d_out)]
            ops += self._wgrad_ops(u, d_out)
            pad_co = -(-cout // 64) * 64
            oH, oW = 2 * lh, 2 * lw
            pw_, ph_, pn_ = d_out_pitches
            views = [ConvSrc(d_out.data_ptr() + 2 * (out_offset + a * ph_ + b * pw_), 2 * pw_, 2 * ph_, pn_, cout, lw, lh, N) for a in (0, 1) for b in (0, 1)]
            dsegs = [(2 * a + b, 1 - th - a, 1 - tw - b, pad_co // 64) for a in (0, 1) for b in (0, 1) for th in (0, 1) for tw in (0, 1)]
            lo = 0
            for (t, c), (dt, acc) in zip(sources, d_sources):
                ops += self._dgrad("%s.dgrad%d" % (name, lo), wname, map_up_dgrad(wshape, lo, lo + c, pad_co), views, dsegs, c, 1, (lw, lh, N), dt,
                                   dense(lh, lw, c), residual=dt if acc else None)
                lo += c
            dec_bwd.append(ops)
            return u

        center = self._act(N, h4, w4, 256)
        d_center = self._buf(N, h4, w4, 256)
        decoder("center", [(pool4, c4)], hp, wpx, 256, center, dense(h4, w4, 256), d_center, dense(h4, w4, 256), [(d_pool4, False)])
        dec0 = self._act(N, h3, w3, 256)
        d_dec0 = self._buf(N, h3, w3, 256)
        # d_enc4 receives the dec0 skip gradient first (plain write), then the max-pool gradient from center is added
        decoder("dec0", [(enc4, c4), (center, 256)], h4, w4, 256, dec0, dense(h3, w3, 256), d_dec0, dense(h3, w3, 256), [(d_enc4, False), (d_center, False)])
        dec1 = self._act(N, h2, w2, 256)
        d_dec1 = self._buf(N, h2, w2, 256)
        decoder("dec1", [(enc3, c3), (dec0, 256)], h3, w3, 256, dec1, dense(h2, w2, 256), d_dec1, dense(h2, w2, 256), [(d_enc3, False), (d_dec0, False)])
        dec2 = self._act(N, h1, w1, 64)
        d_dec2 = self._buf(N, h1, w1, 64)
        decoder("dec2", [(enc2, c2), (dec1, 256)], h2, w2, 64, dec2, dense(h1, w1, 64), d_dec2, dense(h1, w1, 64), [(d_enc2, False), (d_dec1, False)])
        dec3 = self._act(N, H2, W2, 128)
        d_dec3 = self._buf(N, H2, W2, 128)
        decoder("dec3", [(enc1, c1), (dec2, 64)], h1, w1, 128, dec3, dense(H2, W2, 128), d_dec3, dense(H2, W2, 128), [(d_enc1, False), (d_dec2, False)])
        Wq = W + 4
        dec4 = self._act(N, H, Wq, 32)
        d_dec4 = self._buf(N, H, Wq, 32)
        padded = (32, Wq * 32, H * Wq * 32)
        decoder("dec4", [(dec3, 128)], H2, W2, 32, dec4, padded, d_dec4, padded, [(d_dec3, False)], out_offset=32)
        for nm, t, shp in (("center", center, (N, h4, w4, 256)), ("dec0", dec0, (N, h3, w3, 256)), ("dec1", dec1, (N, h2, w2, 256)),
                           ("dec2", dec2, (N, h1, w1, 64)), ("dec3", dec3, (N, H2, W2, 128)), ("dec4", dec4, (N, H, Wq, 32))):
            self.feats[nm] = (t, shp)
            self.relu_outs[nm] = (t, shp)

        # dec5: plain 3x3 on the W-padded dec4 buffer (window view), relu in the epilogue
        y5 = self._act(N, H, W, 32)
        d_y5 = self._buf(N, H, W, 32)
        src5 = ConvSrc(dec4.data_ptr(), 32, Wq * 32, H * Wq * 32, 128, W, H, N, self._plane(dec4))
        u5 = self._add_unit("dec5", "dec5.block.weight", map_window3_fwd(tuple(P["dec5.block.weight"].shape)), [src5],
                            [(0, kh - 1, 0, 2) for kh in range(3)], 32, 1, (W, H, N), y5, dense(H, W, 32), relu=True)
        self.feats["dec5"] = (y5, (N, H, W, 32))
        self.relu_outs["dec5"] = (y5, (N, H, W, 32))
        self.logits = self._buf(N, self.C, H, W, dtype=torch.float32)
        self.fwd_ops.append(("final_fwd_split" if self.strict else "final_fwd", y5, self.logits))
        self.final_acc = self._buf(self.C * 32 + 8, dtype=torch.float64)

        ops5 = [("final_bwd", self._hi(y5), d_y5), ("relu_bwd", d_y5, None, self._hi(y5), d_y5)]
        ops5 += self._wgrad_ops(u5, d_y5)
        ops5 += self._dgrad("dec5.dgrad", "dec5.block.weight", map_conv_dgrad(u5.wshape, pad_co_to=64), [_src_dense(d_y5, N, H, W, 32)],
                            [(0, kh - 1, kw - 1, 1) for kh in range(3) for kw in range(3)], 32, 1, (W, H, N), d_dec4, padded, out_offset=32)

        # ---- backward program: head, decoder (reverse), pool4 fan-in, encoder (reverse)
        self.bwd_ops = [("zero_grads",)] + ops5
        for ops in reversed(dec_bwd):
            self.bwd_ops += ops
        # enc4's gradient = dec0 skip gradient (already in d_enc4) + max-pool backward of the center branch
        d_enc4_pool = self._buf(N, h4, w4, c4)
        self.bwd_ops.append(("maxpool_bwd_split" if self.strict else "maxpool_bwd", enc4, d_pool4, d_enc4_pool, N, h4, w4, c4, 2, 2, 0))
        self.bwd_ops.append(("relu_bwd", d_enc4, d_enc4_pool, None, d_enc4))  # plain sum (no mask)
        for ops in reversed(bwd):
            self.bwd_ops += ops
        self.bwd_ops.append(("unpack_all",))
        self._mean = (ctypes.c_float * 3)(0.485, 0.456, 0.406)
        self._std = (ctypes.c_float * 3)(0.229, 0.224, 0.225)

    # ---------------------------------------------------------------- GPU executor
    def _run(self, ops, x=None, dlogits=None):
        lib = _lib.load()
        st = _lib.current_stream_ptr()
        P = self.params
        for op in ops:
            k = op[0]
            if k == "conv":
                op[1].run(st)
            elif k == "pack_all":
                self._run_pack_all(lib, st)
                for w, m, d, scale, single in self.split_pack_list:
                    n = d.shape[1]
                    _lib.check((lib.rsb_pack_weights1_split if single else lib.rsb_pack_weights_split)(
                        P[w].data_ptr(), m.data_ptr(), d.data_ptr(), n, n, scale, self.overflow.data_ptr(), st), "rsb_pack_weights_split[%s]" % w)
            elif k == "unpack_all":
                # packed weight gradients (fp32 arena chunks) -> the flat OIHW gradient buffer: one launch per chunk
                if self._unpack_all is None:
                    self._grad(self.unpack_list[0][2])
                    self._unpack_all = []
                    deterministic = os.environ.get("RSB_WGRAD_DETERMINISTIC", "1") != "0"
                    for ci, (chunk, used) in enumerate(self._dw_chunks):
                        gmap = torch.full((used, 4), -1, dtype=torch.int32, device=self.device)
                        for dwp, m, wname, c, off in self.unpack_list:
                            if c == ci:
                                gmap[off:off + m.shape[0]] = torch.where(m >= 0, m + self._grad_offset[wname], m)
                        if deterministic:
                            # invert the scatter map once: every OIHW gradient element gathers its <= 4 packed contributions in order
                            flat = gmap.reshape(-1).long()
                            valid = flat >= 0
                            src = flat[valid]
                            pk = (torch.arange(flat.numel(), device=self.device) // 4)[valid]
                            order = torch.argsort(src, stable=True)
                            src, pk = src[order], pk[order]
                            uniq, counts = torch.unique_consecutive(src, return_counts=True)
                            assert int(counts.max()) <= 4, "a weight receives more than 4 packed gradient contributions"
                            start = torch.cumsum(counts, 0) - counts
                            gid = torch.repeat_interleave(torch.arange(uniq.numel(), device=self.device), counts)
                            rank = torch.arange(src.numel(), device=self.device) - start[gid]
                            inv = torch.full((uniq.numel(), 4), -1, dtype=torch.int32, device=self.device)
                            inv[gid, rank] = pk.int()
                            self._unpack_all.append(("gather", uniq.int().contiguous(), inv.contiguous(), chunk))
                            del gmap
                        else:
                            self._unpack_all.append(("scatter", gmap, None, chunk, used))
                for item in self._unpack_all:
                    if item[0] == "gather":
                        _, dst_idx, inv, chunk = item
                        _lib.check(lib.rsb_unpack_grads_gather(chunk.data_ptr(), dst_idx.data_ptr(), inv.data_ptr(), self._grads_flat.data_ptr(),
                                                               dst_idx.numel(), 1.0 / self.loss_scale, st), "rsb_unpack_grads_gather")
                    else:
                        _, gmap, _, chunk, used = item
                        _lib.check(lib.rsb_unpack_grads(chunk.data_ptr(), gmap.data_ptr(), self._grads_flat.data_ptr(), used, 1.0 / self.loss_scale, st), "rsb_unpack_grads")
            elif k == "bn_stats":
                # batch sums + (in the reduction's last block) statistics, folded scale/shift and the running-stat update
                b = op[1]
                pf = b.prefix
                if b.partials is not None:
                    _lib.check(lib.rsb_bn_partials_finalize(b.partials.data_ptr(), b.partial_rows, b.sums.data_ptr(), P[pf + ".weight"].data_ptr(),
                                                            P[pf + ".bias"].data_ptr(), P[pf + ".running_mean"].data_ptr(),
                                                            P[pf + ".running_var"].data_ptr(), P[pf + ".num_batches_tracked"].data_ptr(),
                                                            b.mean.data_ptr(), b.invstd.data_ptr(), b.scale.data_ptr(), b.shift.data_ptr(), b.M, b.C,
                                                            BN_EPS, BN_MOMENTUM, 1 if BN_CHAINED else 0, st), "rsb_bn_partials_finalize")
                    continue
                _lib.check((lib.rsb_bn_stats_finalize_chained if BN_CHAINED else lib.rsb_bn_stats_finalize)(b.z.data_ptr(), b.sums.data_ptr(), P[pf + ".weight"].data_ptr(), P[pf + ".bias"].data_ptr(),
                                                     P[pf + ".running_mean"].data_ptr(), P[pf + ".running_var"].data_ptr(),
                                                     P[pf + ".num_batches_tracked"].data_ptr(), b.mean.data_ptr(), b.invstd.data_ptr(),
                                                     b.scale.data_ptr(), b.shift.data_ptr(), b.M, b.C, BN_EPS, BN_MOMENTUM, st), "rsb_bn_stats_finalize_chained")
            elif k == "bn_finalize":
                pass  # fused into the bn_stats launch (kept as an op for the CPU emulation of the plan)
            elif k == "bn_stats_split":
                b = op[1]
                pf = b.prefix
                _lib.check((lib.rsb_bn_stats_finalize_split_chained if BN_CHAINED else lib.rsb_bn_stats_finalize_split)(
                    b.zpair.data_ptr(), b.zplane, b.sums.data_ptr(), P[pf + ".weight"].data_ptr(), P[pf + ".bias"].data_ptr(),
                    P[pf + ".running_mean"].data_ptr(), P[pf + ".running_var"].data_ptr(), P[pf + ".num_batches_tracked"].data_ptr(),
                    b.mean.data_ptr(), b.invstd.data_ptr(), b.scale.data_ptr(), b.shift.data_ptr(), b.M, b.C, BN_EPS, BN_MOMENTUM,
                    self.overflow.data_ptr(), st), "rsb_bn_stats_finalize_split")
            elif k == "bn_apply_split":
                _, b, res, y, relu = op
                _lib.check((lib.rsb_bn_apply_split_chained if BN_CHAINED else lib.rsb_bn_apply_split)(
                    b.zpair.data_ptr(), b.zplane, b.scale.data_ptr(), b.shift.data_ptr(), res.data_ptr() if res is not None else None,
                    self._plane(res), y.data_ptr(), self._plane(y), b.M, b.C, 1 if relu else 0, st), "rsb_bn_apply_split")
            elif k == "bn_apply":
                _, b, res, y, relu = op
                _lib.check((lib.rsb_bn_apply_chained if BN_CHAINED else lib.rsb_bn_apply)(b.z.data_ptr(), b.scale.data_ptr(), b.shift.data_ptr(), res.data_ptr() if res is not None else None,
                                            y.data_ptr(), b.M, b.C, 1 if relu else 0, st), "rsb_bn_apply")
            elif k == "bn_bwd":
                _, b, dy, y, dz, g = op
                pf = b.prefix
                # y = half(relu(z*scale + shift)) with no identity branch: the mask is re-derived from z, y is not read
                zmask = y is not None and getattr(b, "plain_relu_y", None) is y
                _lib.check((lib.rsb_bn_backward_chained if BN_CHAINED else lib.rsb_bn_backward)(dy.data_ptr(), y.data_ptr() if (y is not None and not zmask) else None, b.z.data_ptr(),
                                               b.mean.data_ptr(), b.invstd.data_ptr(), P[pf + ".weight"].data_ptr(),
                                               b.scale.data_ptr() if zmask else None, b.shift.data_ptr() if zmask else None,
                                               b.sums.data_ptr(), dz.data_ptr(), g.data_ptr() if g is not None else None,
                                               self._grad(pf + ".weight").data_ptr(), self._grad(pf + ".bias").data_ptr(), 1.0 / self.loss_scale,
                                               b.M, b.C, st), "rsb_bn_backward")
            elif k == "relu_bwd":
                _, a, b2, y, out = op
                _lib.check(lib.rsb_relu_backward(a.data_ptr(), b2.data_ptr() if b2 is not None else None, y.data_ptr() if y is not None else None,
                                                 out.data_ptr(), a.numel(), st), "rsb_relu_backward")
            elif k == "maxpool":
                _, src, dst, n, h, w, c, kk, s, p = op
                _lib.check(lib.rsb_maxpool_nhwc(src.data_ptr(), dst.data_ptr(), n, h, w, c, kk, s, p, st), "rsb_maxpool_nhwc")
            elif k in ("maxpool_bwd", "maxpool_bwd_split"):
                _, xx, dy, dx, n, h, w, c, kk, s, p = op
                scratch = self._pool_scratch.get(id(dx))
                if scratch is None:
                    scratch = self._pool_scratch[id(dx)] = torch.empty(dy.numel(), dtype=torch.uint8, device=dx.device)
                if k == "maxpool_bwd_split":
                    _lib.check(lib.rsb_maxpool_backward_split(xx.data_ptr(), self._plane(xx), dy.data_ptr(), dx.data_ptr(), scratch.data_ptr(),
                                                              n, h, w, c, kk, s, p, st), "rsb_maxpool_backward_split")
                    continue
                _lib.check(lib.rsb_maxpool_backward(xx.data_ptr(), dy.data_ptr(), dx.data_ptr(), scratch.data_ptr(), n, h, w, c, kk, s, p, st),
                           "rsb_maxpool_backward")
            elif k == "maxpool_split":
                _, src, dst, n, h, w, c, kk, s, p = op
                _lib.check(lib.rsb_maxpool_nhwc_split(src.data_ptr(), self._plane(src), dst.data_ptr(), self._plane(dst), n, h, w, c, kk, s, p, st),
                           "rsb_maxpool_nhwc_split")
            elif k == "wgrad":
                _, u, dy = op
                if not hasattr(u, "wgrad_plan"):
                    u.wgrad_plan = ctypes.c_void_p()
                    _lib.check(lib.rsb_wgrad_plan_create(ctypes.byref(u.wdesc), dy.data_ptr() + 2 * u.out_offset, u.dw_packed.data_ptr(),
                                                         ctypes.byref(u.wgrad_plan)), "rsb_wgrad_plan_create[%s]" % u.name)
                    self._wgrad_scratch_for(u.wgrad_plan)
                _lib.check(lib.rsb_wgrad_run(u.wgrad_plan, st), "rsb_wgrad_run[%s]" % u.name)
            elif k == "prepass":
                kind = 0 if x.dtype == torch.float32 else 1
                _lib.check(lib.rsb_prepass_s2d(x.data_ptr(), kind, self.s2d.data_ptr(), self.N, self.H, self.W, self._mean, self._std, st), "rsb_prepass_s2d")
            elif k == "prepass_split":
                kind = 0 if x.dtype == torch.float32 else 1
                _lib.check(lib.rsb_prepass_s2d_split(x.data_ptr(), kind, self.s2d.data_ptr(), self._plane(self.s2d), self.N, self.H, self.W,
                                                     self._mean, self._std, st), "rsb_prepass_s2d_split")
            elif k == "final_fwd_split":
                _, y5, logits = op
                _lib.check(lib.rsb_final_forward_split(y5.data_ptr(), self._plane(y5), P["final.weight"].data_ptr(), P["final.bias"].data_ptr(),
                                                       self.overflow.data_ptr(), logits.data_ptr(), self.N, self.H * self.W, self.C, st),
                           "rsb_final_forward_split")
            elif k == "final_fwd":
                _, y5, logits = op
                _lib.check(lib.rsb_final_forward(y5.data_ptr(), P["final.weight"].data_ptr(), P["final.bias"].data_ptr(), logits.data_ptr(),
                                                 self.N, self.H * self.W, self.C, st), "rsb_final_forward")
            elif k == "final_bwd":
                _, y5, d_y5 = op
                _lib.check(lib.rsb_final_backward(dlogits.data_ptr(), y5.data_ptr(), P["final.weight"].data_ptr(), d_y5.data_ptr(), self.final_acc.data_ptr(),
                                                  self._grad("final.weight").data_ptr(), self._grad("final.bias").data_ptr(), self.loss_scale,
                                                  self.N, self.H * self.W, self.C, st), "rsb_final_backward")
            elif k == "zero_grads":
                self._grad("final.bias")
                self._grads_flat.zero_()
            else:  # pragma: no cover
                raise AssertionError(k)

    def _run_pack_all(self, lib, st):
        """fp32 master weights -> every fp16 operand layout of every layer. The packed buffers are slices of a few arena
        chunks; when all weights sit in one parameter arena (offsets from the lowest address fit in int32, e.g. the flat arena
        of robosat_b200.optim.Adam) ONE launch per chunk fills them through a combined map, else one launch per layout."""
        P = self.params
        ptrs = tuple(P[w].data_ptr() for w, _, _, _, _ in self.pack_list)
        if self._pack_all is None or self._pack_all["ptrs"] != ptrs:
            base = min(ptrs)
            span = max((p - base) // 4 + P[e[0]].numel() for p, e in zip(ptrs, self.pack_list))
            combined = None
            if span < 2 ** 31 and all((p - base) % 4 == 0 for p in ptrs):
                combined = []
                for ci, (chunk, used) in enumerate(self._pack_chunks):
                    gmap = torch.full((used, 4), -1, dtype=torch.int32, device=self.device)
                    kinds = []  # (offset, one source per element?) per layout of this chunk, in address order
                    for p, (w, m, d, c, off) in zip(ptrs, self.pack_list):
                        if c == ci:
                            gmap[off:off + m.shape[0]] = torch.where(m >= 0, m + int((p - base) // 4), m)
                            kinds.append((off, bool((m[:, 1:] < 0).all())))
                    # runs of layouts with a single source per element (everything but the pre-summed nearest-x2 taps) go through
                    # the 1-index kernel: 4 instead of 16 map bytes per element (layout offsets are multiples of 8 elements)
                    kinds.sort()
                    runs = []
                    for off, single in kinds:
                        if runs and runs[-1][2] == single:
                            continue
                        if runs:
                            runs[-1][1] = off
                        runs.append([off, used, single])
                    for start, end, single in runs:
                        m = gmap[start:end, 0].contiguous() if single else gmap[start:end].contiguous()
                        combined.append((m, chunk[start:end], end - start, single))
            self._pack_all = {"ptrs": ptrs, "combined": combined, "base": base}
        if self._pack_all["combined"] is None:
            for w, m, d, _, _ in self.pack_list:
                _lib.check(lib.rsb_pack_weights(P[w].data_ptr(), m.data_ptr(), d.data_ptr(), d.numel(), st), "rsb_pack_weights")
            return
        for gmap, chunk, used, single in self._pack_all["combined"]:
            _lib.check((lib.rsb_pack_weights1 if single else lib.rsb_pack_weights)(self._pack_all["base"], gmap.data_ptr(), chunk.data_ptr(), used, st),
                       "rsb_pack_weights")

    # ---------------------------------------------------------------- CUDA-graph replay of the two op lists
    # A step is ~520 launches of mostly 10-40 us kernels; replaying each op list from one CUDA graph removes the launch gaps
    # between them (16.2 -> 15.5 ms for forward + backward at 16 x 512^2, profiles/r2_train.md). The lists only touch static
    # buffers; what varies per call (the input tensor, dlogits) is copied into a static buffer first, and everything baked into
    # kernel arguments at capture time (parameter addresses, the loss scale) is part of the graph's key: a change re-captures.
    def _graph_key(self, static):
        return (static.data_ptr(), float(self.loss_scale), tuple(v.data_ptr() for v in self.params.values()))

    def _replay(self, which, ops, src, **kw):
        """run `ops` with the per-call tensor `src` through the graph of list `which` ("fwd" / "bwd"); the first two calls of a
        key run eagerly (lazy tables are built there), the third captures."""
        slot = self._graphs.setdefault((which, src.dtype, tuple(src.shape)), {"static": torch.empty_like(src), "calls": 0, "graph": None, "key": None})
        static = slot["static"]
        static.copy_(src)
        key = self._graph_key(static)
        if slot["key"] != key:
            slot.update(key=key, calls=0, graph=None)
        name = "x" if which == "fwd" else "dlogits"
        if slot["graph"] is None:
            slot["calls"] += 1
            if slot["calls"] <= 2 or torch.cuda.is_current_stream_capturing():
                self._run(ops, **{name: static}, **kw)
                return
            graph = torch.cuda.CUDAGraph()
            try:
                with torch.cuda.graph(graph, capture_error_mode="thread_local"):
                    self._run(ops, **{name: static}, **kw)
            except Exception as exc:  # noqa: BLE001 -- a failed capture leaves the eager path, loudly
                import warnings

                warnings.warn("robosat_b200: CUDA-graph capture of the training %s plan failed (%r); running it kernel by kernel" % (which, exc))
                self.use_graph = False
                torch.cuda.synchronize()
                self._run(ops, **{name: static}, **kw)
                return
            slot["graph"] = graph
        slot["graph"].replay()

    def forward(self, x):
        if self.plan_only:
            raise _lib.RsbError("UNetTrainEngine was built with plan_only=True; there is no CPU execution path")
        assert x.is_cuda and x.is_contiguous()
        if self.use_graph:
            self._replay("fwd", self.fwd_ops, x)
        else:
            self._run(self.fwd_ops, x=x)
        if self.strict and not torch.cuda.is_current_stream_capturing():
            # the pack's overflow count travels to the host behind the forward; overflowed() reads it without a synchronisation
            if self._overflow_host is None:
                self._overflow_host = torch.zeros(1, dtype=torch.int32, pin_memory=True)
                self._overflow_event = torch.cuda.Event()
            self._overflow_host.copy_(self.overflow, non_blocking=True)
            self._overflow_event.record()
        return self.logits

    def overflowed(self):
        """strict precision: True once a finished forward has counted packed weights past their layer's exponent (the weights grew
        beyond the headroom fixed when the plan was built; that step's gradients are not finite). Never synchronises: the answer
        trails the stream by the forwards that have not completed yet. The owner then builds a new plan (fresh exponents)."""
        if not self.strict or self._overflow_event is None or not self._overflow_event.query():
            return False
        return int(self._overflow_host[0]) > 0

    def accumulate_into(self, targets):
        """targets: {parameter name: fp32 contiguous .grad tensor}. Adds this step's gradients into them with ONE kernel
        (what autograd's per-tensor AccumulateGrad would do in ~170 launches). The segment table is cached per set of
        destination pointers."""
        names = [n for n in targets if n in self.grads]
        key = tuple((n, targets[n].data_ptr()) for n in names)
        cached = self._accum_tables.get(key)
        if cached is None:
            rows, seg = [], 16384
            for n in names:
                g, t = self.grads[n], targets[n]
                assert t.dtype == torch.float32 and t.is_contiguous() and t.numel() == g.numel() and t.device == g.device, n
                for off in range(0, g.numel(), seg):
                    rows.append((g.data_ptr() + 4 * off, t.data_ptr() + 4 * off, min(seg, g.numel() - off)))
            table = torch.tensor(rows, dtype=torch.int64).reshape(-1, 3).to(self.device)
            self._accum_tables.clear()
            cached = self._accum_tables[key] = (table, len(rows))
        table, nrows = cached
        _lib.check(_lib.load().rsb_multi_axpy(table.data_ptr(), nrows, 1.0, _lib.current_stream_ptr()), "rsb_multi_axpy")

    def backward(self, dlogits):
        """dlogits: fp32 [N, C, H, W] gradient of the loss w.r.t. the logits (unscaled). Fills self.grads."""
        if self.plan_only:
            raise _lib.RsbError("UNetTrainEngine was built with plan_only=True; there is no CPU execution path")
        assert dlogits.is_cuda and dlogits.is_contiguous() and dlogits.dtype == torch.float32
        self._grad("final.bias")
        if self.use_graph:
            self._replay("bwd", self.bwd_ops, dlogits)
        else:
            self._run(self.bwd_ops, dlogits=dlogits)
        return self.grads
