"""Benchmark of the RoboSat segmentation hot path on B200 (BASELINE.json).

    python bench.py [--gpus N --steps K --warmup W] [--impl reference] [--dump-outputs DIR]
    torchrun ... bench.py --gpus N ...           (one rank per GPU, NCCL)

Prints ONE JSON line (rank 0). --dump-outputs DIR writes what the last timed step of each precision returned (rank 0) as
DIR/<precision>_logits.npy and DIR/<precision>_bins.npy, so that two builds can be compared output for output.

Headline = BASELINE.json configs[1] (`rs predict`: ResNet50-UNet, 2 classes, synthetic 3x512x512 tiles, batch 32 per GPU) in the
STRICT precision -- the mode whose outputs meet the parity contract (logits 1e-3 rel, argmax identical up to the fp32 noise
floor; tests/test_unet_gpu.py). One "step" = one tile batch through the whole path (pre-pass, 56 convolution launches, 2
max-pools, softmax/crop/quantise head).
    value      tiles/s, inputs resident in HBM, CUDA events around K steps, max over ranks
    e2e        tiles/s through the public host API (TilePredictor.submit/collect: pinned host uint8 tiles in, uint8 bins out;
               both copies inside the timed region)
    roofline   executed tensor FLOP/s of the dominant convolution instantiation (timed alone -> against the BURST bf16 peak
               of MEASURED_PEAKS.json; the sustained fraction and the whole-step rate are printed beside it)
    fast       the same three for the fast precision (single fp16 operands, logits ~2e-3): labelled secondary
    cpu_baseline  the UNMODIFIED reference (oracle/_ref, torch CPU fp32) on a bounded sample of the workload (N=1 only)
Other BASELINE configs, each a sub-record measured at the N the run was launched with:
    train      configs[2]: rs train step (2-class, Lovasz, 3x512x512, batch 16 per GPU) incl. the gradient all-reduce
    train_cfg5 configs[4]: 6-class, 3x1024x1024, batch 8 per GPU, data-parallel over N GPUs (ms in NCCL vs compute)
    cfg4       configs[3]: a synthetic slippy-map PNG directory sharded over the ranks through the real `rs predict` shard
               loop (decode -> halo stitch -> net -> PNG), end-to-end tiles/s and the stage that bounds it
`--impl reference` times the unmodified reference alone (rank 0), same metric / config.
"""

import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TILE = 512
BATCH = 32
CLASSES = 2
FWD_GFLOP_DENSE = 167.160  # per 3x512x512 tile, dense-equivalent (SURVEY.md 8(d), BASELINE.md 3)
TRAIN_GFLOP_DENSE = {(2, 512): 500.246, (6, 1024): 2001.790}  # fwd + bwd per tile (SURVEY.md 8(d))
WORKLOAD = "rs predict: ResNet50-UNet, 2-class, 3x512x512 synthetic tiles, batch=32 per GPU"
METRIC = "512x512 tiles/sec (predict fwd)"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"tflops_sustained": d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "tflops_burst": d.get("bf16_tflops"),
                "hbm_gbs": d.get("hbm_gbs"), "src": "measured"}
    return {"tflops_sustained": 1400.0, "tflops_burst": 1590.0, "hbm_gbs": 6650.0, "src": "fallback"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 100 ms while the timed region runs."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------------
# reference arm: the unmodified reference on the host cores
# ----------------------------------------------------------------------------------------------------------------------
def host_threads():
    """cores this process can really use: min(affinity mask, cgroup CPU quota)"""
    from robosat_b200.hostinfo import usable_cores

    return usable_cores()


def cpu_reference_leg(steps, warmup, tiles_per_step, threads=None):
    """The reference's own predict step on the CPU, through its public classes, unmodified (oracle/_ref):
    `net = DataParallel(UNet(2)); outputs = net(images); probs = softmax(outputs, 1).data.cpu().numpy()` (predict.py:47-87).
    Falls back to the oracle restatement (kind "port") only when oracle/_ref is not installed."""
    import torch

    from robosat_b200 import synth

    sd = synth.make_state_dict(CLASSES, seed=0)
    kind = "reference"
    try:
        from baseline import ref_loader

        net = ref_loader.reference_net(sd, CLASSES)

        def run(x):
            with torch.no_grad():
                return torch.nn.functional.softmax(net(x), dim=1).data.cpu().numpy()
    except ImportError:
        from oracle import unet_oracle

        kind = "port"

        def run(x):
            return unet_oracle.predict_probs(sd, x).numpy()

    # torchrun exports OMP_NUM_THREADS=1: ask for the cores this process may run on, explicitly. More threads than the box can
    # really schedule (cgroup quotas, SMT) make oneDNN slower, not faster, so the thread count is the fastest of a few candidates
    # on a quick 256x256 probe -- the reference gets its best host configuration, not the nominal one.
    avail = host_threads()
    if threads is None:
        probe = synth.normalize_tiles(synth.make_tiles_u8(2, 256, seed=2))
        best = None
        for t in sorted({avail, max(1, avail // 2), max(1, avail // 4), min(avail, 32), min(avail, 16), min(avail, 8)}, reverse=True):
            torch.set_num_threads(t)
            run(probe)
            t0 = time.perf_counter()
            run(probe)
            dt = time.perf_counter() - t0
            if best is None or dt < best[0]:
                best = (dt, t)
        threads = best[1]
    torch.set_num_threads(threads)
    cores = torch.get_num_threads()
    x = synth.normalize_tiles(synth.make_tiles_u8(tiles_per_step, TILE, seed=1))
    for _ in range(warmup):
        run(x)
    t0 = time.perf_counter()
    for _ in range(steps):
        run(x)
    dt = time.perf_counter() - t0
    return {"value": steps * tiles_per_step / dt, "unit": "tiles/s", "cores": cores, "kind": kind,
            "sample": "%d steps x %d tiles of 3x%dx%d through the unmodified reference (robosat.unet.UNet + softmax, torch CPU fp32), %d threads "
                      "(fastest of the candidates <= %d available)" % (steps, tiles_per_step, TILE, TILE, cores, avail)}, dt / steps


def cpu_baseline_subprocess(steps=2, warmup=1, tiles_per_step=16):
    """cpu_baseline of the GPU arm: `bench.py --impl reference` on a bounded sample (3 x 16 tiles, 10-30 s of CPU work) in a
    child process that cannot see the GPUs."""
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="")
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE", "OMP_NUM_THREADS"):
        env.pop(k, None)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", str(steps), "--warmup", str(warmup),
                          "--tiles-per-step", str(tiles_per_step)], env=env, capture_output=True, text=True, timeout=900)
    for ln in reversed(out.stdout.strip().splitlines()):
        if ln.startswith("{"):
            return json.loads(ln)["cpu_baseline"]
    raise RuntimeError("reference arm printed no JSON: " + out.stderr[-300:])


def reference_gpu_leg(dev, steps=3, warmup=2):
    """Secondary (SURVEY.md 8(d) "optional secondary"): the UNMODIFIED reference with a visible GPU -- `nn.DataParallel(UNet)`
    moves itself to cuda:0 and runs torch eager / cuDNN (TF32 convolutions by default): the existing Blackwell path. Timed host
    to host like predict.py:83-87 (fp32 NCHW tiles in, fp32 probabilities out), batch 32. Not the CPU baseline, not our code."""
    import torch

    from baseline import ref_loader
    from robosat_b200 import synth

    sd = synth.make_state_dict(CLASSES, seed=0)
    net = ref_loader.reference_net(sd, CLASSES)
    x = synth.normalize_tiles(synth.make_tiles_u8(BATCH, TILE, seed=1))

    def run():
        with torch.no_grad():
            return torch.nn.functional.softmax(net(x.to(dev)), dim=1).data.cpu().numpy()

    for _ in range(warmup):
        run()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = time.perf_counter() - t0
    del net
    torch.cuda.empty_cache()
    return {"value": steps * BATCH / dt, "unit": "tiles/s", "kind": "unmodified reference on cuda:0 (torch %s eager, cuDNN, allow_tf32=%s)" % (
        torch.__version__, torch.backends.cudnn.allow_tf32), "steps": steps, "batch": BATCH,
            "note": "host to host incl. H2D of fp32 tiles and D2H of fp32 probabilities, as predict.py:83-87 does"}


def run_reference(args, rank):
    if rank != 0:
        return
    # The reference's CPU path: on a host with a visible GPU `nn.DataParallel` moves the module to cuda:0 by itself (a one-GPU
    # DataParallel calls module.to(device)), so the GPUs are hidden from THIS process before torch initialises CUDA -- exactly
    # the situation of `cuda = false` on a GPU-less host (predict.py:47-63), where DataParallel is a pass-through.
    os.environ["CUDA_VISIBLE_DEVICES"] = ""
    # a step is a bounded sample of the workload's batch: up to its 32 tiles, shrunk so that the whole run stays within ~400
    # tiles (about 3 minutes at the 2-3 tiles/s the host cores reach; the per-tile CPU rate does not depend on the batch size
    # beyond a few tiles). The sample actually used is stated in cpu_baseline.sample.
    per_step = args.tiles_per_step or max(1, min(BATCH, 400 // max(1, args.steps + args.warmup)))
    cb, s_per_step = cpu_reference_leg(args.steps, args.warmup, per_step)
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "tiles/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": bench_config(args.gpus),
            "cpu_baseline": cb, "e2e": {"value": cb["value"], "unit": "tiles/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def bench_config(world):
    return {"workload": WORKLOAD, "global_batch": world * BATCH, "parallelism": "tile shards, dp%d, 1 weight broadcast" % world,
            "l2": "inputs rotate over 4 batches; per-step activations (2.5 - 5 GB) >> 126 MB L2"}


# ----------------------------------------------------------------------------------------------------------------------
# predict leg (configs[1]) for one precision
# ----------------------------------------------------------------------------------------------------------------------
def layer_profile(engine, x, reps=3):
    """Per-launch device times (CUDA events on the launch stream, each launch alone) and executed FLOPs."""
    import torch

    from robosat_b200 import _lib

    stream = _lib.current_stream_ptr()
    engine.forward(x)
    torch.cuda.synchronize()
    mult = 3 if engine.strict else 1  # strict precision issues hi*lo, lo*hi and hi*hi for every K step
    rows = []
    for op in engine.ops:
        if op[0] != "conv":
            continue
        c = op[1]
        d = c.desc
        # executed MACs: every output pixel-phase x Cout x K (padded K blocks and tile padding are executed too,
        # but only the algorithmic part is counted as useful work)
        if hasattr(d, "taps_h"):  # line-buffer plan
            K, phases, kern = d.taps_h * d.taps_w * d.cin, d.nsub * d.nphase_a, "conv_row_kernel<%d,%d,%d>" % (32 if d.cin == 32 else 64, d.Cout, d.mode)
        else:
            K, phases = 64 * sum(d.segs[i].cblocks for i in range(d.nseg)), d.phases
            kern = "conv_tc_kernel<%d,%d,%d,%d,%d>" % (d.block_n, d.mode, 1 if d.residual else 0, d.cta_pair, d.split)
        flops = 2.0 * mult * d.Nt * d.Ht * d.Wt * phases * d.Cout * K
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for a, b in evs:
            a.record()
            c.run(stream)
            b.record()
        torch.cuda.synchronize()
        ms = min(a.elapsed_time(b) for a, b in evs)
        rows.append({"name": c.name, "kernel": kern, "block_n": getattr(d, "block_n", d.Cout), "mode": d.mode, "ms": ms, "gflop": flops / 1e9,
                     "tflops": flops / ms / 1e9, "tiles": c.info()["tiles"], "kblocks": c.info()["kblocks"]})
    return rows


DUMP_PIXELS = 1 << 20  # of the 8.4 M output pixels of a batch: 12 MB per precision instead of 96 MB


def dump_outputs(out_dir, precision, logits, bins):
    """Writes what one predict step hands its caller -- fp32 logits [N, C, H, W] and the uint8 foreground bins [N, H, W] --
    at the same DUMP_PIXELS pixels, drawn once with a fixed seed: <precision>_logits.npy [DUMP_PIXELS, C] and
    <precision>_bins.npy [DUMP_PIXELS], both float32."""
    import numpy as np
    import torch

    n, c, h, w = logits.shape
    pix = torch.randperm(n * h * w, generator=torch.Generator().manual_seed(0))[:DUMP_PIXELS].sort().values.to(logits.device)
    os.makedirs(out_dir, exist_ok=True)
    sampled = {"logits": logits.reshape(n, c, h * w)[pix // (h * w), :, pix % (h * w)], "bins": bins.reshape(-1)[pix]}
    for name, t in sampled.items():
        np.save(os.path.join(out_dir, "%s_%s.npy" % (precision, name)), t.float().cpu().numpy())


def predict_leg(precision, sd, dev, rank, world, steps, warmup, dist, with_clocks, layers_out=None, dump_dir=None):
    import torch

    from robosat_b200 import synth
    from robosat_b200.predictor import TilePredictor

    pred = TilePredictor(sd, CLASSES, BATCH, TILE, overlap=0, device=dev, precision=precision)
    n_in = 4  # rotate distinct input batches; activations (GBs per step) already exceed the 126 MB L2 many times over
    inputs = [synth.make_tiles_u8(BATCH, TILE, seed=100 + rank * 10 + i).to(dev) for i in range(n_in)]
    qbuf = torch.empty((BATCH, TILE, TILE), dtype=torch.uint8, device=dev)

    def step(i):
        pred.quantize(pred.logits(inputs[i % n_in]), qbuf)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(k):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for i in range(k):
            step(i)
        e1.record()
        barrier()
        return e0.elapsed_time(e1)

    # nvidia-smi needs ~1 s to start reporting and samples every 100 ms: the sampler covers warm-up and the timed K steps,
    # all of them the same back-to-back step
    sampler = ClockSampler(dev.index)
    if rank == 0 and with_clocks:
        sampler.start()
        time.sleep(1.0)
    for i in range(warmup):
        step(i)
    barrier()
    ms = timed(steps)
    clocks = sampler.stop() if rank == 0 and with_clocks else None
    if clocks is not None:
        clocks["window"] = "warm-up + the %d timed steps" % steps
    if dump_dir and rank == 0:
        dump_outputs(dump_dir, precision, pred.engine.logits, qbuf)

    # end to end through the host API: pinned host tiles in, uint8 bins out, copies inside the timed region
    host_batches = [synth.make_tiles_u8(BATCH, TILE, seed=200 + rank * 10 + i).pin_memory() for i in range(2)]
    for i in range(3):
        pred.predict_u8(host_batches[i % 2])
    barrier()
    t0 = time.perf_counter()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    acc = 0
    for i in range(steps):
        pred.submit(host_batches[i % 2])
        if i >= 1:
            acc += int(pred.collect()[0, 0, 0])
    acc += int(pred.collect()[0, 0, 0])
    e3.record()
    barrier()
    e2e_ms = e2.elapsed_time(e3)
    wall_ms = (time.perf_counter() - t0) * 1e3

    vals = [ms, e2e_ms, wall_ms]
    if world > 1:
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vals = t.tolist()
    ms, e2e_ms, wall_ms = vals

    out = {"precision": precision, "ms": ms, "e2e_ms": e2e_ms, "wall_ms": wall_ms, "clocks": clocks, "launches": pred.num_launches(),
           "h2d": pred.h2d_bytes, "d2h": pred.d2h_bytes}
    if rank == 0:
        pk = peaks()
        rows = layer_profile(pred.engine, inputs[0])
        by_kernel = {}
        for r in rows:
            a = by_kernel.setdefault(r["kernel"], {"ms": 0.0, "gflop": 0.0, "launches": 0})
            a["ms"] += r["ms"]
            a["gflop"] += r["gflop"]
            a["launches"] += 1
        dom = max(by_kernel, key=lambda k: by_kernel[k]["ms"])
        dk = by_kernel[dom]
        conv_ms = sum(r["ms"] for r in rows)
        conv_gflop = sum(r["gflop"] for r in rows)
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tpath):  # DRAM bytes per launch of the dominant kernel from the committed ncu --set full capture
            ent = json.load(open(tpath)).get("kernels", {}).get(dom)
            if ent:
                traffic = {"value": ent["mb_per_launch"], "unit": "MB per launch (ncu dram read+write)",
                           "source": "profiles/ncu_traffic.json (committed ncu --set full capture, not re-measured in this run)"}
        achieved = dk["gflop"] / dk["ms"]
        step_tf = conv_gflop / (ms / steps)  # executed FLOPs of all convolutions / whole-step time (incl. pools, head, launch gaps)
        out["roofline"] = {
            "bound": "tensor", "kernel": dom, "achieved": achieved, "peak": pk["tflops_burst"], "unit": "TFLOP/s", "frac": achieved / pk["tflops_burst"],
            "traffic": traffic, "peak_source": pk["src"] + " bf16 BURST (the kernel is timed alone, min of 3 launches)",
            "frac_of_sustained_peak": achieved / pk["tflops_sustained"], "launches_per_step": dk["launches"], "ms_per_step": dk["ms"],
            "all_conv_tflops_isolated": conv_gflop / conv_ms, "all_conv_ms_isolated": conv_ms,
            "step": {"tflops": step_tf, "peak": pk["tflops_sustained"], "frac": step_tf / pk["tflops_sustained"],
                     "note": "executed conv FLOPs / whole-step time vs the measured SUSTAINED bf16 peak"},
            "flops": "executed (sub-pixel decoder: 100.7 GFLOP/tile instead of the 167.16 dense-equivalent%s)" % (
                "; strict precision executes 3 MMAs per K step = 302.2 GFLOP/tile" if precision == "strict" else ""),
            "by_kernel": {k: {"ms_per_step": round(v["ms"], 4), "launches": v["launches"], "tflops": round(v["gflop"] / v["ms"], 1)}
                          for k, v in sorted(by_kernel.items(), key=lambda kv: -kv[1]["ms"])}}
        if layers_out:
            with open(layers_out.replace(".json", "_%s.json" % precision), "w") as fp:
                json.dump({"layers": rows, "by_kernel": by_kernel}, fp, indent=1)
    del pred, inputs, host_batches
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------------------------------------------------
# training legs (configs[2], configs[4]): data parallel, one all-reduce of the flat gradient arena per step
# ----------------------------------------------------------------------------------------------------------------------
def train_leg(dev, rank, world, dist, classes, size, batch, steps, warmup, label):
    """One step = zero_grad + train-mode forward + Lovasz loss + backward (+ NCCL all-reduce of the flat fp32 gradient arena
    when N > 1) + Adam, through the public module API -- exactly the body of `_epoch` in robosat_b200/tools/train.py."""
    import torch

    from robosat_b200 import synth
    from robosat_b200.dist import allreduce_sum_
    from robosat_b200.losses import LovaszLoss2d
    from robosat_b200.optim import Adam
    from robosat_b200.unet import UNet

    net = torch.nn.DataParallel(UNet(classes, pretrained=False), device_ids=[dev.index]).to(dev)
    net.load_state_dict(synth.make_state_dict(classes, seed=0))
    opt = Adam(net.parameters(), lr=1e-4)
    opt.mark_used([not n.startswith("module.resnet.fc.") for n, _ in net.named_parameters()])
    crit = LovaszLoss2d().to(dev)
    xs = [synth.normalize_tiles(synth.make_tiles_u8(batch, size, seed=300 + 10 * rank + i)).to(dev) for i in range(2)]
    ms_ = [synth.make_masks(batch, size, classes, seed=310 + 10 * rank + i).to(dev) for i in range(2)]
    net.train()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(steps + warmup)]

    def step(i):
        opt.zero_grad()
        loss = crit(net(xs[i % 2]), ms_[i % 2])
        (loss / world if world > 1 else loss).backward()
        ev[i][0].record()
        allreduce_sum_(opt.flat_grad, world)
        ev[i][1].record()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(warmup):
        step(i)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(warmup, warmup + steps):
        loss = step(i)
    e1.record()
    barrier()
    total = e0.elapsed_time(e1)
    nccl = sum(ev[i][0].elapsed_time(ev[i][1]) for i in range(warmup, warmup + steps))
    vals = [total, nccl]
    if world > 1:
        t = torch.tensor(vals, device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        vals = t.tolist()
    total, nccl = vals
    grad_mb = opt.flat_grad.numel() * 4 / 1e6
    last = float(loss.detach())
    del net, opt, xs, ms_
    torch.cuda.empty_cache()
    dense = TRAIN_GFLOP_DENSE.get((classes, size))
    out = {"metric": "%dx%d tiles/sec (train fwd+bwd, Lovasz, Adam)" % (size, size), "value": world * batch * steps / (total / 1e3), "unit": "tiles/s",
           "n_gpus": world, "ms_per_step": total / steps, "steps": steps, "warmup": warmup, "batch_per_gpu": batch, "config": label,
           "collective": {"op": "ncclAllReduce(sum) of the flat fp32 gradient arena, one call per step after backward()" if world > 1 else "none (N=1)",
                          "mbytes": grad_mb, "ms_per_step": nccl / steps, "share_of_step": nccl / total,
                          "busbw_gbs": (2.0 * (world - 1) / world * grad_mb / 1e3) / (nccl / steps / 1e3) if world > 1 and nccl > 0 else None},
           "compute_ms_per_step": (total - nccl) / steps, "last_loss": last}
    if dense:
        out["dense_equiv_tflops_per_gpu"] = batch * steps * dense / total
        out["frac_of_sustained_peak_dense_equiv"] = out["dense_equiv_tflops_per_gpu"] / peaks()["tflops_sustained"]
    return out


# ----------------------------------------------------------------------------------------------------------------------
# configs[3]: slippy-map directory through the real `rs predict` shard loop
# ----------------------------------------------------------------------------------------------------------------------
def cfg4_leg(dev, rank, world, dist, sd, tiles_per_gpu, batch=32, tile=512, overlap=32):
    """Every rank writes its own 1/N of a contiguous x/y grid of synthetic PNG tiles (untimed), then -- barrier -- runs
    `robosat_b200.tools.predict.run_shard` on its shard of the whole directory: enumerate, decode (once per tile, prefetched on
    pool threads), halo stitch on the device, U-Net (strict precision), quantise, PNG encode + write. Timed: barrier -> all
    ranks done; tiles/s = all tiles / that time. The real tool shards 100 k tiles; the benchmark uses `tiles_per_gpu` per GPU
    so that it finishes in seconds -- stated in the record."""
    import argparse as ap

    import torch

    from robosat_b200 import synth
    from robosat_b200.tools.predict import run_shard

    root = os.environ.get("RSB_CFG4_DIR") or os.path.join(tempfile.gettempdir(), "rsb_cfg4_%s" % os.environ.get("MASTER_PORT", "single"))
    tiles_dir, probs_dir = os.path.join(root, "tiles"), os.path.join(root, "probs")
    cols = max(1, tiles_per_gpu // 32)  # 32 rows (y) x `cols` columns (x) per rank: shard_range on the (z, x, y)-sorted list = this block
    def all_ok(ok, what):
        """a failure on ONE rank (disk full, bad tile) must not leave the others waiting in a collective: every phase ends
        with an all-reduce of an ok flag and all ranks leave together"""
        flag = torch.tensor([1.0 if ok else 0.0], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if flag.item() < 1.0:
            if rank == 0:
                shutil.rmtree(root, ignore_errors=True)
            raise RuntimeError("cfg4 leg: %s failed on at least one rank%s" % (what, "" if ok else " (this one: %s)" % err[0]))

    err = [None]
    try:
        if rank == 0:
            shutil.rmtree(root, ignore_errors=True)
            os.makedirs(tiles_dir, exist_ok=True)
    except Exception as exc:
        err[0] = repr(exc)
    all_ok(err[0] is None, "creating the scratch directory")
    threads = max(4, host_threads() // world)
    t0 = time.perf_counter()
    try:
        synth.write_slippy_tiles(tiles_dir, 18, range(1000 + rank * cols, 1000 + (rank + 1) * cols), range(2000, 2032), size=tile, seed=7 + rank, workers=threads)
    except Exception as exc:
        err[0] = repr(exc)
    gen_s = time.perf_counter() - t0
    args = ap.Namespace(batch_size=batch, overlap=overlap, tile_size=tile, workers=0, tiles=tiles_dir, probs=probs_dir)
    os.environ["RSB_QUIET"] = "1"
    # warm-up (untimed, like the W steps of the other legs): the same loop over a 64-tile directory of this rank's own, so that
    # lazy imports, CUDA module loading, the thread pools' first start and the page cache of the codec are not in the timed run.
    # Every timed run still builds its plans, lists the directory and allocates its buffers (setup_s in the record).
    if err[0] is None:
        try:
            warm_root = os.path.join(root, "warm%d" % rank)
            synth.write_slippy_tiles(os.path.join(warm_root, "tiles"), 18, range(500, 502), range(2000, 2032), size=tile, seed=99 + rank, workers=threads)
            wargs = ap.Namespace(batch_size=batch, overlap=overlap, tile_size=tile, workers=0, tiles=os.path.join(warm_root, "tiles"),
                                 probs=os.path.join(warm_root, "probs"))
            run_shard(0, 1, wargs, dev, sd, CLASSES, stats={})
            shutil.rmtree(warm_root, ignore_errors=True)
        except Exception as exc:
            err[0] = repr(exc)
    torch.cuda.synchronize()
    all_ok(err[0] is None, "writing the synthetic tiles")  # doubles as the barrier before the timed region
    t0 = time.perf_counter()
    st = None
    try:
        st = run_shard(rank, world, args, dev, sd, CLASSES, stats={})
        torch.cuda.synchronize()
    except Exception as exc:
        err[0] = repr(exc)
    mine = time.perf_counter() - t0
    all_ok(st is not None, "the shard loop")
    keys = ["wall_s", "decode_wait_s", "gpu_wait_s", "png_drain_s", "png_cpu_s", "setup_s"]
    vec = torch.tensor([mine] + [float(st.get(k, 0.0)) for k in keys] + [float(st["tiles"])], device=dev, dtype=torch.float64)
    mx = vec.clone()
    sm = vec.clone()
    if world > 1:
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(sm, op=dist.ReduceOp.SUM)
    total_tiles = int(sm[-1].item())
    wall = mx[0].item()
    # device time of the network alone at this shape, for the stage table
    from robosat_b200.predictor import TilePredictor

    pred = TilePredictor(sd, CLASSES, batch, tile + 2 * overlap, overlap=overlap, device=dev)
    xin = pred.device_input()
    xin.random_(0, 256)
    q = torch.empty((batch, tile, tile), dtype=torch.uint8, device=dev)
    for _ in range(3):
        pred.quantize(pred.logits(xin), q)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        pred.quantize(pred.logits(xin), q)
    e1.record()
    torch.cuda.synchronize()
    net_ms = e0.elapsed_time(e1) / 5
    del pred
    torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()
    if rank == 0:
        shutil.rmtree(root, ignore_errors=True)
    setup = mx[6].item()
    loop_s = max(wall - setup, 1e-9)
    net_s = st["batches"] * net_ms / 1e3
    blocked = {"decode_wait_s": mx[2].item(), "gpu_wait_s": mx[3].item(), "png_drain_s": mx[4].item()}
    host = dict(st.get("main_thread_s", {}))
    # what bounds the steady-state loop: the device if the network's own time fills >= 80 % of it, else the largest host item
    if net_s >= 0.8 * loop_s:
        bound = "net: the U-Net on the device (%.1f ms per batch of %d at %dx%d) fills %.0f %% of the loop" % (net_ms, batch, tile + 2 * overlap, tile + 2 * overlap, 100 * net_s / loop_s)
    else:
        cand = {"PNG decode (main thread waiting for rsb_png_read_rgb_batch, %d threads per rank)" % st.get("decode_threads", 0): blocked["decode_wait_s"],
                "PNG encode backlog at the end (rsb_png_write_p8_batch, %d threads per rank)" % st["pool_threads"]: blocked["png_drain_s"],
                "host launch path (ctypes launches of %d kernels per batch)" % 60: host.get("launch_s", 0.0),
                "host bookkeeping of the stitch step (slot tables, upload calls)": host.get("stitch_s", 0.0) - blocked["decode_wait_s"]}
        bound = max(cand, key=cand.get)
    return {"metric": "512x512 tiles/sec end to end (rs predict: PNG tiles in -> probability PNGs out)", "value": total_tiles / wall, "unit": "tiles/s",
            "steady_state_tiles_per_s": total_tiles / loop_s, "setup_s": setup,
            "setup_note": "directory listing + plan construction (fold/split/pack 39 M weights) + buffers: paid once per run, amortised over 100 k tiles",
            "n_gpus": world, "tiles": total_tiles, "tiles_per_gpu": total_tiles // world, "wall_s": wall, "batch": batch, "tile_size": tile, "overlap": overlap,
            "precision": "strict", "host_threads_per_rank": threads,
            "config": "rs predict: ResNet50-UNet, 2-class, 3x512x512 (+32 px halo), synthetic slippy-map PNG dir sharded across %d x B200 "
                      "(%d tiles here; BASELINE cfg 4 names 100k)" % (world, total_tiles),
            "stages_max_over_ranks": {"main_thread_blocked": blocked, "main_thread_loop_rank0": host, "codec_wall_s_rank0": st.get("png_cpu_s"),
                                      "net_device_s": net_s, "net_ms_per_batch_576": net_ms, "input_generation_s_untimed": gen_s},
            "bound": bound, "gpu_only_tiles_per_s": world * batch / (net_ms / 1e3)}


# ----------------------------------------------------------------------------------------------------------------------
def serve_leg(dev, requests=100, warmup=10, size=512):
    """`rs serve` request latency (SURVEY.md 8(f) row 3; serve.py:135-172): one 3x512x512 tile per call through
    `SegmentEngine.run` -- pinned uint8 H2D, normalise, U-Net, argmax, uint8 D2H, host sync -- replayed as one CUDA graph,
    and the same kernels launched one by one on the stream. Secondary figure beside the headline."""
    import torch

    from robosat_b200 import synth
    from robosat_b200.serve import SegmentEngine

    sd = synth.make_state_dict(2, seed=0)
    tiles = synth.make_tiles_u8(4, size, seed=5).numpy()
    threads = torch.get_num_threads()
    torch.set_num_threads(1)  # the CPU-baseline leg leaves 100+ OpenMP workers spinning; a request is single-threaded host work
    out = {"metric": "rs serve latency per 512x512 tile (batch 1, host to host, strict precision)", "unit": "ms", "requests": requests}
    for key, use_graph in (("graph_ms", True), ("stream_ms", False)):
        eng = SegmentEngine(sd, 2, size, size, device=dev, use_graph=use_graph)
        if use_graph and eng.graph is None:
            out["graph_error"] = eng.graph_error
            continue
        h_in = eng.h_in.numpy()
        for i in range(warmup):
            h_in[0] = tiles[i % 4]
            eng.run()
        t0 = time.perf_counter()
        for i in range(requests):
            h_in[0] = tiles[i % 4]
            eng.run()
        out[key] = (time.perf_counter() - t0) * 1e3 / requests
        del eng, h_in
        torch.cuda.empty_cache()
    torch.set_num_threads(threads)
    return out


def stitch_leg(dev, batch=32, size=512, overlap=32, reps=50):
    """Halo stitch on the device (SURVEY.md 8(f) row 1; tiles.py:162-227): one `rsb_stitch_halo` launch builds the buffered
    batch uint8 [32][576][576][3] from the device tile cache. HBM-bound byte work: algorithmic bytes = canvas read + written."""
    import torch

    from robosat_b200 import _lib

    lib = _lib.load()
    F = size + 2 * overlap
    store = torch.randint(0, 256, (9 * batch, size, size, 3), dtype=torch.uint8, device=dev)
    table = torch.arange(9 * batch, dtype=torch.int32, device=dev).reshape(batch, 9).contiguous()
    out = torch.empty((batch, F, F, 3), dtype=torch.uint8, device=dev)
    st = _lib.current_stream_ptr()
    for _ in range(3):
        _lib.check(lib.rsb_stitch_halo(store.data_ptr(), table.data_ptr(), out.data_ptr(), batch, size, overlap, st), "rsb_stitch_halo")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        _lib.check(lib.rsb_stitch_halo(store.data_ptr(), table.data_ptr(), out.data_ptr(), batch, size, overlap, st), "rsb_stitch_halo")
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    gbps = 2 * out.numel() / ms / 1e6
    return {"metric": "halo stitch of 32 buffered 576x576 tiles on the device", "ms_per_batch": ms, "achieved_gbps": gbps,
            "peak_gbps": peaks()["hbm_gbs"], "frac": gbps / peaks()["hbm_gbs"], "tiles_per_s": batch / ms * 1e3}


def guarded(fn, *a, **kw):
    """secondary legs must never take the headline down with them"""
    try:
        return fn(*a, **kw)
    except Exception as exc:
        import traceback

        return {"error": "%s: %s" % (type(exc).__name__, exc), "trace": traceback.format_exc()[-600:]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-train", action="store_true", help="skip the training legs (configs[2], configs[4])")
    ap.add_argument("--no-cfg4", action="store_true", help="skip the slippy-map directory leg (configs[3])")
    ap.add_argument("--no-extras", action="store_true", help="headline + fast mode only")
    ap.add_argument("--cfg4-tiles", type=int, default=0, help="tiles per GPU in the synthetic slippy-map directory (0: 2048 up to 2 GPUs, 512 beyond)")
    ap.add_argument("--tiles-per-step", type=int, default=0, help="(--impl reference) tiles per step instead of the automatic bounded sample")
    ap.add_argument("--layers-out", default=None, help="write the per-layer timing tables (JSON) here (_strict / _fast suffix)")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR", help="(--impl ours) write the outputs of the last timed step of each precision here (.npy)")
    args = ap.parse_args()
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes the outputs of the timed predict path of --impl ours; --impl reference has none to write")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference(args, rank)

    import torch
    import torch.distributed as dist

    from robosat_b200 import synth

    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "1")
        # NCCL prints its version banner to STDOUT when the communicator is created if NCCL_DEBUG is VERSION / WARN (the GPU boxes
        # export it): stdout must carry the one JSON line only, so the communicator is created here with fd 1 pointed at stderr.
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.all_reduce(torch.zeros(1, device=dev))
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)

    # weights: rank 0 materialises the checkpoint; ONE NCCL broadcast of the flat fp32 state_dict (the predict path's only collective)
    sd = synth.make_state_dict(CLASSES, seed=0)
    if world > 1:
        from robosat_b200.dist import broadcast_state_dict

        sd = broadcast_state_dict(sd if rank == 0 else None, template=sd, device=dev)  # rank 0 is the only one whose copy is used

    strict = predict_leg("strict", sd, dev, rank, world, args.steps, args.warmup, dist, True, args.layers_out, args.dump_outputs)
    fast = predict_leg("fast", sd, dev, rank, world, args.steps, args.warmup, dist, False, args.layers_out, args.dump_outputs)

    extras = {}
    if not args.no_extras:
        if not args.no_train:
            extras["train"] = guarded(train_leg, dev, rank, world, dist, 2, 512, 16, 8, 3,
                                      "rs train: ResNet50-UNet, 2-class, Lovasz loss, 3x512x512 synthetic tiles+masks, batch=16 per GPU, %dxB200" % world)
            extras["train_cfg5"] = guarded(train_leg, dev, rank, world, dist, 6, 1024, 8, 5, 3,
                                           "rs train: ResNet50-UNet, 6-class, 3x1024x1024 synthetic, batch=8/GPU, data parallel over %dxB200 NVLink" % world)
        if not args.no_cfg4:
            # 2 048 tiles (1.4 GB of PNGs) per GPU up to two GPUs, 512 beyond: the scratch directory lives under the temp dir
            per_gpu = args.cfg4_tiles if args.cfg4_tiles > 0 else (2048 if world <= 2 else 512)
            extras["cfg4"] = guarded(cfg4_leg, dev, rank, world, dist, sd, per_gpu)

    line = None
    if rank == 0:
        tiles = world * BATCH * args.steps

        def summary(r):
            s = {"value": tiles / (r["ms"] / 1e3), "unit": "tiles/s", "ms_per_step": r["ms"] / args.steps,
                 "e2e": {"value": tiles / (r["e2e_ms"] / 1e3), "unit": "tiles/s", "h2d_bytes_per_step": r["h2d"], "d2h_bytes_per_step": r["d2h"],
                         "wall_ms": r["wall_ms"], "api": "TilePredictor.submit/collect (pinned uint8 in, uint8 bins out)"},
                 "roofline": r.get("roofline")}
            return s

        s, f = summary(strict), summary(fast)
        line = {"metric": METRIC, "value": s["value"], "unit": "tiles/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": s["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f16 hi+lo operand pairs (3 MMAs per K step), fp32 accumulate: strict precision, meets the parity contract",
                "data": "synthetic", "config": bench_config(world), "precision": "strict",
                "dense_equiv_tflops": s["value"] * FWD_GFLOP_DENSE / 1e3,
                "e2e": s["e2e"], "gpu_launches": world * args.steps * strict["launches"], "clocks": strict["clocks"], "roofline": s["roofline"],
                "fast": dict(f, precision="fast", dtype="f16 operands (1 MMA per K step), fp32 accumulate",
                             note="secondary: logits ~2e-3 rel, ~0.1 % argmax flips at near-ties -- does NOT meet the parity contract",
                             dense_equiv_tflops=f["value"] * FWD_GFLOP_DENSE / 1e3)}
        line.update(extras)
        if world == 1 and not args.no_extras:
            if not args.no_cpu_baseline:  # the CPU baseline is an N=1 figure (rank 0 only), ~10-30 s of CPU work
                line["cpu_baseline"] = guarded(cpu_baseline_subprocess)
            line["reference_cudnn"] = guarded(reference_gpu_leg, dev)
            line["stitch"] = guarded(stitch_leg, dev)
            line["serve"] = guarded(serve_leg, dev)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return line


if __name__ == "__main__":
    main()
