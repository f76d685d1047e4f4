"""Training-step throughput (BASELINE.json configs[2]: ResNet50-UNet, 2 classes, Lovasz loss, 3x512x512, batch 16, 1 GPU).
One step = zero_grad + forward (train-mode BN) + Lovasz loss + backward + Adam, through the public module API.

    python scripts/bench_train.py [--batch 16 --size 512 --steps 10 --warmup 3 --precision fast|strict]

--precision sets UNet.train_precision (fast: single fp16 forward; strict: hi/lo fp16 forward, robosat_b200/train_engine.py).
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from robosat_b200 import synth  # noqa: E402
from robosat_b200.losses import LovaszLoss2d  # noqa: E402
from robosat_b200.optim import Adam  # noqa: E402
from robosat_b200.unet import UNet  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--precision", choices=("fast", "strict"), default="fast")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    net = torch.nn.DataParallel(UNet(2, pretrained=False), device_ids=[0]).to(dev)
    net.load_state_dict(synth.make_state_dict(2, seed=0))
    net.module.train_precision = args.precision
    opt = Adam(net.parameters(), lr=1e-4)
    opt.mark_used([not n.startswith("module.resnet.fc.") for n, _ in net.named_parameters()])
    crit = LovaszLoss2d().to(dev)
    xs = [synth.normalize_tiles(synth.make_tiles_u8(args.batch, args.size, seed=10 + i)).to(dev) for i in range(2)]
    ms = [synth.make_masks(args.batch, args.size, 2, seed=20 + i).to(dev) for i in range(2)]
    net.train()
    ev = {k: [] for k in ("fwd", "loss", "bwd", "adam")}

    def step(i, timed):
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(5)]
        opt.zero_grad()
        marks[0].record()
        out = net(xs[i % 2])
        marks[1].record()
        loss = crit(out, ms[i % 2])
        marks[2].record()
        loss.backward()
        marks[3].record()
        opt.step()
        marks[4].record()
        if timed:
            torch.cuda.synchronize()
            for j, k in enumerate(("fwd", "loss", "bwd", "adam")):
                ev[k].append(marks[j].elapsed_time(marks[j + 1]))
        return loss

    for i in range(args.warmup):
        step(i, False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    losses = []
    for i in range(args.steps):
        losses.append(step(i, False))
    e1.record()
    torch.cuda.synchronize()
    total = e0.elapsed_time(e1)
    for i in range(3):
        step(i, True)
    out = {"metric": "512x512 tiles/sec (train fwd+bwd+Lovasz+Adam)", "value": args.batch * args.steps / (total / 1e3), "unit": "tiles/s",
           "precision": args.precision, "ms_per_step": total / args.steps, "batch": args.batch, "size": args.size, "steps": args.steps,
           "breakdown_ms": {k: sum(v) / len(v) for k, v in ev.items()}, "loss_first": float(losses[0]), "loss_last": float(losses[-1]),
           "fwd_bwd_dense_tflops": args.batch * args.steps * 500.246 / (total / 1e3) / 1e3,
           "gpu": torch.cuda.get_device_name(dev)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
