"""Timing aid (not a test): receiver noise in the fused launch (noise_std= / noise_seed=, VR_FLAG_NOISE) against the same
per-sequence route without noise, and against adding the noise in torch, in one process, alternating the variants.

Variants of every workload (NTU shape: T = 300, 25 joints, 2 bodies; one placement per sequence, a third at the origin):
  noise   the per-sequence route with noise_std (N,) = 0.5 and a 0-d int64 seed tensor: the noise is added inside the launch;
  clean   the same call without the noise keywords (per-sequence placements, no noise);
  torch   the alternative without this feature: the synthesis-only launch writes the I/Q (N, T, 2) (what forward_debug
          saves), torch adds torch.randn * sigma sqrt(1/2), and the general-kernel STFT (tcgen05 GEMM) transforms it.
Workloads:
  1. forward at N = 4096 and 16384 (noise, clean, torch);
  2. forward_image(x, 256) at N = 4096;
  3. forward_upsampled(x, 250, 3, image_size=256) at N = 148 (x raw);
  4. forward_views at R = 4, 16384 outputs;
  5. forward + backward of out.square().mean() with trainable placements at N = 4096 (noise, clean, torch).

Each workload is timed in --rounds rounds, the variants alternating, each round K steps between CUDA events after warm-up; the
median and the range over the rounds are printed, and noise/clean and noise/torch of the medians.  The card's name, power
limit and max SM clock are read in the same run.
Usage: python tools/bench_noise.py [--rounds R] [--steps K] [--out FILE]"""
import argparse
import json
import math
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from skeleton_action_recognition_b200 import VirtualRadar, _cabi  # noqa: E402
from skeleton_action_recognition_b200.layers.virtual_radar import _SynthFunction  # noqa: E402
from tools.bench_radar_views import placements, step_alloc, timed  # noqa: E402
from tools.bench_upsampled_backward import card  # noqa: E402

SIGMA = 0.5


def workloads():
    """-> (name, {variant: step}); a step returns the output."""
    g = torch.Generator().manual_seed(7)
    seed = torch.tensor(1234, dtype=torch.int64, device="cuda")

    def variants(N, T=300, R=None, call=None, grad=False, alternative=False):
        layer = VirtualRadar(wavelength=1e-3, device="cuda:0").to("cuda:0")
        x = (torch.randn(N, 3, T, 25, 2, generator=g) * 0.4).cuda()
        lam, loc = placements(N, R or 1, g)
        lam, loc = (lam, loc) if R else (lam.reshape(N), loc.reshape(N, 3))
        if grad:
            lam.requires_grad_(True)
            loc.requires_grad_(True)
        std = torch.full(lam.shape, SIGMA, device="cuda")
        kw = {} if call is None else call

        def run(**nkw):
            if R:
                out = layer.forward_views(x, loc, lam, **kw, **nkw)
            elif "num_pad_frames" in kw:
                out = layer.forward_upsampled(x, kw["num_pad_frames"], kw["sigma"], kw.get("image_size"),
                                              radar_location=loc, wavelength=lam, **nkw)
            elif "image_size" in kw:
                out = layer.forward_image(x, kw["image_size"], radar_location=loc, wavelength=lam, **nkw)
            else:
                out = layer(x, radar_location=loc, wavelength=lam, **nkw)
            if grad:
                lam.grad = loc.grad = None
                out.square().mean().backward()
            return out

        def run_torch():
            if grad:
                iq = _SynthFunction.apply(lam, loc, x, layer, _cabi.VR_FLAG_PER_SEQUENCE)
            else:
                iq = layer._synth(x, _cabi.VR_FLAG_PER_SEQUENCE, lam, loc)
            iq = iq + torch.randn(iq.shape, device="cuda") * (std * math.sqrt(0.5))[:, None, None]
            out = layer.stft.logmag(iq)
            if grad:
                lam.grad = loc.grad = None
                out.square().mean().backward()
            return out

        v = {"noise": lambda: run(noise_std=std, noise_seed=seed), "clean": run}
        if alternative:
            v["torch"] = run_torch
        return v

    for N in (4096, 16384):
        yield "forward N=%d" % N, variants(N, alternative=True)
    yield "forward_image S=256 N=4096", variants(4096, call=dict(image_size=256))
    yield "forward_upsampled k=250 S=256 N=148", variants(148, call=dict(num_pad_frames=250, sigma=3, image_size=256))
    yield "forward_views R=4 N=4096 (16384 outputs)", variants(4096, R=4)
    yield "fwd+bwd placements N=4096", variants(4096, grad=True, alternative=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lines = ["card (name, power limit, max SM clock): %s" % card(),
             "median over %d rounds of %d steps (min..max), the variants alternating; alloc: peak bytes a step allocates "
             "beyond its inputs" % (args.rounds, args.steps)]
    print(lines[0], "\n" + lines[1], flush=True)
    res = {}
    for name, var in workloads():
        with torch.set_grad_enabled(name.startswith("fwd+bwd")):
            for _ in range(2):                               # warm-up (plans, caches, allocator)
                for fn in var.values():
                    fn()
            alloc = {v: step_alloc(fn) for v, fn in var.items()}
            t = {v: [] for v in var}
            for _ in range(args.rounds):
                for v, fn in var.items():
                    t[v].append(timed(fn, args.steps))
        res[name] = {"ms": t, "alloc_bytes": alloc}
        med = {v: statistics.median(t[v]) for v in t}
        lines.append(name)
        for v in var:
            lines.append("    %-6s %9.3f ms (%.3f..%.3f)  alloc %8.1f MB" % (v, med[v], min(t[v]), max(t[v]), alloc[v] / 1e6))
        ratio = "    noise/clean %.3f" % (med["noise"] / med["clean"])
        if "torch" in med:
            ratio += "  noise/torch %.3f" % (med["noise"] / med["torch"])
        lines.append(ratio)
        print("\n".join(lines[-(len(var) + 2):]), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n" + json.dumps(res) + "\n")


if __name__ == "__main__":
    main()
