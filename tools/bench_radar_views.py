"""Timing aid (not a test): R radar views per sequence (VirtualRadar.forward_views, VR_FLAG_VIEWS) against the per-sequence
route on the repeated batch, in one process, alternating the variants.

Variants of every workload (NTU shape: T = 300, 25 joints, 2 bodies; R distinct placements per sequence, a third of them at
the origin; N sequences, N R outputs):
  views      layer.forward_views(x, loc (N, R, 3), lam (N, R)), x of N sequences;
  repeated   layer(xr, radar_location=loc (N R, 3), wavelength=lam (N R,)), xr = x.repeat_interleave(R, 0) built beforehand;
  +repeat    the same, with the repeat_interleave inside the timed step.
Workloads:
  1. forward at N R = 4096 and 16384 outputs, R = 1, 2, 4, 8;
  2. forward_image(x, 256) at N R = 4096, R = 4;
  3. forward_upsampled(x, 250, 3, image_size=256) at N R = 148, R = 4 (x raw; the spline is solved for N or N R sequences);
  4. forward + backward of out.square().mean() with trainable placements, (N, R) / (N, R, 3) gradients, N R = 4096, R = 4,
     without and with dL/dx (the backward's two view layouts: units per output, or per x row with the views in order).

Each workload is timed in --rounds rounds, the variants alternating, each round K steps between CUDA events after warm-up; the
median and the range over the rounds are printed.  `alloc` is the peak memory a step allocates beyond what was allocated
before it (outputs, the repeated x of +repeat, autograd buffers); `x` the input the variant reads.  For the forward, `GB/s`
is the bytes the step must move at least -- each x sequence read once (180 000 B) and each spectrogram written once
(19 456 B) -- over its time; the repeated variants read R times as much x.  The card's name, power limit and max SM clock are
read in the same run.
Usage: python tools/bench_radar_views.py [--rounds R] [--steps K] [--out FILE]"""
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
X_BYTES, OUT_BYTES = 3 * 300 * 25 * 2 * 4, 256 * 19 * 4


def placements(N, R, g):
    lam = torch.tensor([[LAMS[(n + r) % 4] for r in range(R)] for n in range(N)], dtype=torch.float32)
    loc = torch.randn(N, R, 3, generator=g) * 1.5
    loc.view(-1, 3)[::3] = 0.0
    return lam.cuda(), loc.cuda()


def workloads():
    """-> (name, N, R, bytes bound or None, {variant: (step, input bytes)}); a step returns the output."""
    g = torch.Generator().manual_seed(5)

    def variants(NR, R, T=300, call=None, grad=False, xgrad=False):
        N = NR // R
        layer = VirtualRadar(wavelength=1e-3, device="cuda:0").to("cuda:0")
        x = (torch.randn(N, 3, T, 25, 2, generator=g) * 0.4).cuda().requires_grad_(xgrad)
        lam, loc = placements(N, R, g)
        if grad:
            lam.requires_grad_(True)
            loc.requires_grad_(True)
        xr = x.detach().repeat_interleave(R, 0).requires_grad_(xgrad)
        kw = {} if call is None else call

        def run_views():
            out = layer.forward_views(x, loc, lam, **kw)
            if grad:
                lam.grad = loc.grad = x.grad = None
                out.square().mean().backward()
            return out

        def run_repeated(xin):
            lr, Lr = lam.reshape(N * R), loc.reshape(N * R, 3)
            if "num_pad_frames" in kw:
                out = layer.forward_upsampled(xin, kw["num_pad_frames"], kw["sigma"], kw.get("image_size"),
                                              radar_location=Lr, wavelength=lr)
            elif "image_size" in kw:
                out = layer.forward_image(xin, kw["image_size"], radar_location=Lr, wavelength=lr)
            else:
                out = layer(xin, radar_location=Lr, wavelength=lr)
            if grad:
                lam.grad = loc.grad = x.grad = xr.grad = None
                out.square().mean().backward()
            return out

        return {"views": (run_views, x.numel() * 4), "repeated": (lambda: run_repeated(xr), xr.numel() * 4),
                "+repeat": (lambda: run_repeated(x.repeat_interleave(R, 0)), x.numel() * 4)}

    for NR in (4096, 16384):
        for R in (1, 2, 4, 8):
            yield "forward", NR // R, R, NR // R * X_BYTES + NR * OUT_BYTES, variants(NR, R)
    yield "forward_image S=256", 1024, 4, None, variants(4096, 4, call=dict(image_size=256))
    yield "forward_upsampled k=250 S=256", 37, 4, None, variants(148, 4, T=300,
                                                                   call=dict(num_pad_frames=250, sigma=3, image_size=256))
    yield "fwd+bwd placements", 1024, 4, None, variants(4096, 4, grad=True)
    yield "fwd+bwd placements and x", 1024, 4, None, variants(4096, 4, grad=True, xgrad=True)


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def step_alloc(fn):
    """Peak bytes one step allocates beyond what is allocated before it."""
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    return torch.cuda.max_memory_allocated() - base


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lines = ["card (name, power limit, max SM clock): %s" % card(),
             "median over %d rounds of %d steps (min..max), the variants alternating; alloc: peak bytes a step allocates "
             "beyond its inputs; x: input bytes the variant reads" % (args.rounds, args.steps)]
    print(lines[0], "\n" + lines[1], flush=True)
    res = {}
    for name, N, R, bound, var in workloads():
        key = "%s N=%d R=%d (%d outputs)" % (name, N, R, N * R)
        with torch.set_grad_enabled(name.startswith("fwd+bwd")):
            for _ in range(2):                               # warm-up (plans, caches, allocator)
                for fn, _ in var.values():
                    fn()
            alloc = {v: step_alloc(fn) for v, (fn, _) in var.items()}
            t = {v: [] for v in var}
            for _ in range(args.rounds):
                for v, (fn, _) in var.items():
                    t[v].append(timed(fn, args.steps))
        res[key] = {"ms": t, "alloc_bytes": alloc, "x_bytes": {v: b for v, (_, b) in var.items()}, "bound_bytes": bound}
        med = {v: statistics.median(t[v]) for v in t}
        lines.append(key)
        for v in var:
            gbs = "  %6.0f GB/s of the byte bound" % (bound / med[v] / 1e6) if bound else ""
            lines.append("    %-9s %9.3f ms (%.3f..%.3f)  alloc %8.1f MB  x %8.1f MB%s" % (
                v, med[v], min(t[v]), max(t[v]), alloc[v] / 1e6, var[v][1] / 1e6, gbs))
        lines.append("    views/repeated %.3f  views/+repeat %.3f" % (med["views"] / med["repeated"], med["views"] / med["+repeat"]))
        print("\n".join(lines[-(len(var) + 2):]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n" + json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
