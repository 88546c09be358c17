"""Timing aid (not a test): the bitwise-reproducible backward against the library of an earlier build (float atomics in the
adjoint overlap-add, the parameter sums and the split-K kernel gradients), in one process, alternating the two.

Workloads (forward + backward per step):
  1. the default layer with trainable radar parameters and dL/dx, NTU shape (T = 300, 25 joints, 2 bodies), N = 256, 4096;
  2. forward_upsampled(x, 250, image_size=256) with both radar parameters trainable, default kernels, N = 16, 64, 256;
  3. train_stft_kernel=True (general kernels, kernel gradients only), T = 300, hop 16, N = 4096, n_fft = 128, 256, 512;
  4. forward_upsampled(x, 250, image_size=256) with trainable kernels and both radar parameters, N = 64.

Both libraries run the same Python layer: the earlier one is loaded beside the current one and swapped in as the binding's
library.  Each workload is timed in R rounds, current and earlier build alternating, each round K steps between CUDA events
after warm-up; the median and the range over the rounds are printed.  Forward outputs are compared bit for bit.  The card's
name and power limit are read in the same run.
Usage: python tools/bench_deterministic_backward.py --parent-lib PATH [--rounds R] [--steps K] [--out FILE]"""
import argparse
import ctypes
import json
import os
import statistics
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from skeleton_action_recognition_b200 import VirtualRadar, _cabi  # noqa: E402
from tools.bench_upsampled_backward import card  # noqa: E402


def load_parent(path):
    """The earlier library with the current binding's argument types (it lacks the symbols added since)."""
    new = _cabi.lib()
    old = ctypes.CDLL(os.path.abspath(path))
    for name in _cabi.SYMBOLS:
        if hasattr(old, name):
            f, g = getattr(new, name), getattr(old, name)
            if f.argtypes is not None:
                g.argtypes = f.argtypes
            g.restype = f.restype
    return old


def workloads():
    g = torch.Generator().manual_seed(3)
    for N in (256, 4096):
        x = (torch.randn(N, 3, 300, 25, 2, generator=g) * 0.4).cuda()
        layer = VirtualRadar(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], train_wavelength=True,
                             train_radar_location=True, device="cuda:0").to("cuda:0")
        yield "default layer, dL/dx + radar params, NTU N=%d" % N, layer, x, True, lambda l, x: l(x)
    for N in (16, 64, 256):
        x = (torch.randn(N, 3, 300, 25, 2, generator=g) * 0.4).cuda()
        layer = VirtualRadar(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], train_wavelength=True,
                             train_radar_location=True, device="cuda:0").to("cuda:0")
        yield ("forward_upsampled k=250 S=256, radar params, N=%d" % N, layer, x, False,
               lambda l, x: l.forward_upsampled(x, 250, image_size=256))
    for n_fft in (128, 256, 512):
        x = (torch.randn(4096, 3, 300, 25, 2, generator=g) * 0.4).cuda()
        layer = VirtualRadar(wavelength=1e-3, train_stft_kernel=True, n_fft=n_fft, device="cuda:0").to("cuda:0")
        yield "general kernels, kernel grads, T=300 N=4096 n_fft=%d" % n_fft, layer, x, False, lambda l, x: l(x)
    x = (torch.randn(64, 3, 300, 25, 2, generator=g) * 0.4).cuda()
    layer = VirtualRadar(wavelength=1e-3, radar_location=[0.3, -0.2, 1.5], train_wavelength=True, train_radar_location=True,
                         train_stft_kernel=True, device="cuda:0").to("cuda:0")
    yield ("forward_upsampled k=250 S=256, general kernels + radar params, N=64", layer, x, False,
           lambda l, x: l.forward_upsampled(x, 250, image_size=256))


def step(layer, x, want_x, fn):
    for p in layer.parameters():
        p.grad = None
    xi = x.requires_grad_(want_x)
    xi.grad = None
    out = fn(layer, xi)
    out.square().mean().backward()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", required=True)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out", default=os.path.join("profiles", "r03c_deterministic_backward.log"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    libs = {"new": _cabi.lib(), "parent": load_parent(args.parent_lib)}
    lines = ["card (name, power limit, max SM clock): %s" % card(),
             "median over %d rounds of %d steps (min..max), the two builds alternating" % (args.rounds, args.steps)]
    print(lines[0], flush=True)
    result = {}
    for name, layer, x, want_x, fn in workloads():
        outs, times = {}, {k: [] for k in libs}
        for k, L in libs.items():                                # warm-up, and the forward outputs of both builds
            _cabi._lib = L
            for _ in range(2):
                outs[k] = step(layer, x, want_x, fn).detach().clone()
        same = torch.equal(outs["new"], outs["parent"])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.rounds):
            for k, L in libs.items():
                _cabi._lib = L
                step(layer, x, want_x, fn)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(args.steps):
                    step(layer, x, want_x, fn)
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / args.steps)
        _cabi._lib = libs["new"]
        med = {k: statistics.median(v) for k, v in times.items()}
        line = "%-72s new %8.3f ms (%.3f..%.3f)  parent %8.3f ms (%.3f..%.3f)  new/parent %.3f  forward bit-equal %s" % (
            name, med["new"], min(times["new"]), max(times["new"]), med["parent"], min(times["parent"]),
            max(times["parent"]), med["new"] / med["parent"], same)
        print(line, flush=True)
        lines.append(line)
        result[name] = {"new_ms": times["new"], "parent_ms": times["parent"], "forward_bit_equal": same}
        del layer, x
        torch.cuda.empty_cache()
    lines.append(json.dumps(result))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
