"""Timing aid (not a test): the backward pass through the temporal up-sampling.

  1. pad_frames backward alone (C ABI vr_pad_frames_backward_f32) at N = 148, T = 300, k = 250, as the rate at which it
     reads dL/d(out) (45 MB per NTU sequence; 6.66 GB per call, far beyond the 126 MB L2);
  2. forward + backward of forward_upsampled(x, 250, 3, image_size=256) with both radar parameters trainable (fused:
     vr_forward_upsampled_debug_f32 + vr_backward_upsampled_params_f32) against the materialising route
     layer.forward_image(pad_frames(x, 250, 3), 256), N in {16, 64, 256}: time per step and peak allocation.

CUDA events around K calls after warm-up; the card's name and power limit are read in the same run.
Usage: python tools/bench_upsampled_backward.py [--out FILE]"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from skeleton_action_recognition_b200 import VirtualRadar, _cabi, pad_frames  # noqa: E402


def timed(fn, warmup=2, iters=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[torch.cuda.current_device()] if q.returncode == 0 else torch.cuda.get_device_name()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    lines = []

    def log(s):
        print(s, flush=True)
        lines.append(s)

    log("card (name, power limit, max SM clock): %s" % card())
    res = {}

    # 1. pad_frames backward alone
    N, T, V, M, k = 148, 300, 25, 2, 250
    g = torch.randn(N, 3, k * T, V, M, device="cuda")
    gx = torch.empty(N, 3, T, V, M, device="cuda")
    L = _cabi.lib()
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def bwd():
        _cabi.check(L.vr_pad_frames_backward_f32(g.data_ptr(), N, T, V, M, k, ctypes.c_float(3.0), gx.data_ptr(), stream))

    ms = timed(bwd, 2, 10)
    nbytes = g.numel() * 4
    res["pad_frames_backward"] = dict(N=N, T=T, k=k, ms=ms, read_GB=nbytes / 1e9, GB_per_s=nbytes / ms * 1e-6)
    log("pad_frames backward N=%d T=%d k=%d: %.3f ms, reads %.2f GB -> %.0f GB/s (DESIGN 4: measured HBM read rate 6520 GB/s)"
        % (N, T, k, ms, nbytes / 1e9, nbytes / ms * 1e-6))
    del g, gx

    # 2. forward + backward with trainable radar parameters: fused vs materialising
    layer = VirtualRadar(wavelength=5e-4, train_wavelength=True, train_radar_location=True, device="cuda:0").to("cuda:0")
    for N in (16, 64, 256):
        x = torch.randn(N, 3, 300, 25, 2, device="cuda") * 0.3
        routes = (("fused", lambda: layer.forward_upsampled(x, 250, 3, image_size=256)),
                  ("materialising", lambda: layer.forward_image(pad_frames(x, 250, 3), 256)))
        for name, fwd in routes:
            def step():
                fwd().mean().backward()
                layer.zero_grad(set_to_none=True)
            step()
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated()
            torch.cuda.reset_peak_memory_stats()
            step()
            torch.cuda.synchronize()
            peak = torch.cuda.max_memory_allocated() - base
            ms = timed(step, 1, 3)
            res["N%d_%s" % (N, name)] = dict(ms_per_step=ms, peak_MB=peak / 1e6)
            log("fwd+bwd forward_upsampled(k=250, image 256), N=%3d %-13s %9.2f ms/step  peak %9.1f MB"
                % (N, name, ms, peak / 1e6))
        del x
    log(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
