"""Timing aid (not a test): per-sequence radar placements (the `radar_location=` / `wavelength=` keywords,
VR_FLAG_PER_SEQUENCE) against the scalar placement of the module parameters, in one process, alternating the two.

Workloads (NTU shape: T = 300, 25 joints, 2 bodies; distinct wavelength and location per sequence, a third at the origin):
  1. forward, N = 256, stream-ordered and with assume_inputs_ready;
  2. forward, N = 4096 and N = 16384;
  3. forward_image(x, 256), N = 4096;
  4. forward_upsampled(x, 250, 3, image_size=256), N = 148;
  5. forward + backward with both radar parameters trainable (scalar: the module's two gradients; per-sequence: (N,) and
     (N, 3) gradients), N = 256 and 4096, and forward_upsampled(x, 250, image_size=256) under grad, N = 16 and 64.

Each workload is timed in R rounds, the two variants alternating, each round K steps between CUDA events after warm-up;
the median and the range over the rounds are printed, with the card's name and power limit read in the same run.
Usage: python tools/bench_per_sequence_radar.py [--rounds R] [--steps K] [--out FILE]"""
import argparse
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from skeleton_action_recognition_b200 import VirtualRadar  # noqa: E402
from tools.bench_upsampled_backward import card  # noqa: E402

LAMS = (5e-4, 9e-4, 1e-3, 5e-3)


def placements(N, g):
    lam = torch.tensor([LAMS[n % 4] for n in range(N)], dtype=torch.float32)
    loc = torch.randn(N, 3, generator=g) * 1.5
    loc[::3] = 0.0
    return lam.cuda(), loc.cuda()


def workloads():
    """-> (name, scalar step, per-sequence step); a step returns the output."""
    g = torch.Generator().manual_seed(5)
    ntu = lambda N: (torch.randn(N, 3, 300, 25, 2, generator=g) * 0.4).cuda()       # noqa: E731

    def fwd(N, ready=False, call=lambda l, x, **kw: l(x, **kw)):
        layer = VirtualRadar(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], device="cuda:0").to("cuda:0")
        layer.assume_inputs_ready = ready
        x = ntu(N)
        lam, loc = placements(N, g)
        return (lambda: call(layer, x)), (lambda: call(layer, x, radar_location=loc, wavelength=lam))

    def bwd(N, call=lambda l, x, **kw: l(x, **kw)):
        layer = VirtualRadar(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], train_wavelength=True,
                             train_radar_location=True, device="cuda:0").to("cuda:0")
        x = ntu(N)
        lam, loc = placements(N, g)
        lam.requires_grad_(True)
        loc.requires_grad_(True)

        def scalar():
            layer.wavelength.grad = layer.radar_location.grad = None
            out = call(layer, x)
            out.square().mean().backward()
            return out

        def per_seq():
            lam.grad = loc.grad = None
            out = call(layer, x, radar_location=loc, wavelength=lam)
            out.square().mean().backward()
            return out
        return scalar, per_seq

    yield ("forward N=256", *fwd(256))
    yield ("forward N=256 assume_inputs_ready", *fwd(256, ready=True))
    yield ("forward N=4096", *fwd(4096))
    yield ("forward N=16384", *fwd(16384))
    yield ("forward_image S=256 N=4096", *fwd(4096, call=lambda l, x, **kw: l.forward_image(x, 256, **kw)))
    yield ("forward_upsampled k=250 S=256 N=148",
           *fwd(148, call=lambda l, x, **kw: l.forward_upsampled(x, 250, 3, 256, **kw)))
    yield ("fwd+bwd radar params N=256", *bwd(256))
    yield ("fwd+bwd radar params N=4096", *bwd(4096))
    ups = lambda l, x, **kw: l.forward_upsampled(x, 250, 3, 256, **kw)     # noqa: E731
    yield ("fwd+bwd forward_upsampled k=250 S=256 N=16", *bwd(16, ups))
    yield ("fwd+bwd forward_upsampled k=250 S=256 N=64", *bwd(64, ups))


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = ["card (name, power limit, max SM clock): %s" % card(),
             "median over %d rounds of %d steps (min..max), the two variants alternating" % (args.rounds, args.steps)]
    print(lines[0], "\n" + lines[1], flush=True)
    res = {}
    for name, scalar, per_seq in workloads():
        with torch.set_grad_enabled(name.startswith("fwd+bwd")):    # the forward workloads run as inference
            for fn in (scalar, per_seq, scalar, per_seq):     # warm-up (plans, caches)
                fn()
            torch.cuda.synchronize()
            t = {"scalar_ms": [], "per_sequence_ms": []}
            for _ in range(args.rounds):
                t["scalar_ms"].append(timed(scalar, args.steps))
                t["per_sequence_ms"].append(timed(per_seq, args.steps))
        res[name] = t
        ms, mp = statistics.median(t["scalar_ms"]), statistics.median(t["per_sequence_ms"])
        line = "%-44s scalar %9.3f ms (%.3f..%.3f)  per-sequence %9.3f ms (%.3f..%.3f)  per-sequence/scalar %.3f" % (
            name, ms, min(t["scalar_ms"]), max(t["scalar_ms"]), mp, min(t["per_sequence_ms"]), max(t["per_sequence_ms"]),
            mp / ms)
        lines.append(line)
        print(line, flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n" + json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
