"""Timing aid (not a test): forward_upsampled with GENERAL STFT kernels, at N in {16, 64, 256}, T = 300, k = 250, image 256.

  1. train_stft_kernel=True and both radar parameters trainable: forward + backward of
     forward_upsampled(x, 250, 3, image_size=256) (iq-only synthesis from the spline's cubics + kept-frames STFT) against
     the materialising composition F.interpolate(layer(pad_frames(x, 250, 3)).unsqueeze(1), 256): time per step and
     peak allocation;
  2. the same pair under no_grad, with trained (perturbed) but frozen kernels;
  3. kernel time of vr_synth_upsampled_f32 against vr_forward_upsampled_debug_f32 (the fused launch with its 256-point
     FFT and spectrogram store, which the general route used before).

CUDA events around K calls after warm-up; the card's name and power limit are read in the same run.
Usage: python tools/bench_upsampled_general.py [--out FILE]"""
import argparse
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from skeleton_action_recognition_b200 import VirtualRadar, _cabi, pad_frames  # noqa: E402
from tools.bench_upsampled_backward import card, timed  # noqa: E402


def perturb(layer, eps=0.02):
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        layer.stft.wsin.add_((eps * torch.randn(layer.stft.wsin.shape, generator=g)).cuda())
        layer.stft.wcos.add_((eps * torch.randn(layer.stft.wcos.shape, generator=g)).cuda())
    return layer


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
    T, k, S = 300, 250, 256
    interp = torch.nn.functional.interpolate
    trainable = VirtualRadar(wavelength=5e-4, train_wavelength=True, train_radar_location=True, train_stft_kernel=True,
                             device="cuda:0").to("cuda:0")
    frozen = perturb(VirtualRadar(wavelength=5e-4, device="cuda:0").to("cuda:0"))
    for N in (16, 64, 256):
        x = torch.randn(N, 3, T, 25, 2, device="cuda") * 0.3
        for mode, layer in (("fwd+bwd", trainable), ("no_grad", frozen)):
            routes = (("new", lambda: layer.forward_upsampled(x, k, 3, image_size=S)),
                      ("materialising", lambda: interp(layer(pad_frames(x, k, 3)).unsqueeze(1), S)))
            for name, fwd in routes:
                if mode == "fwd+bwd":
                    def step():
                        fwd().mean().backward()
                        layer.zero_grad(set_to_none=True)
                else:
                    def step():
                        with torch.no_grad():
                            fwd()
                step()
                torch.cuda.synchronize()
                base = torch.cuda.memory_allocated()
                torch.cuda.reset_peak_memory_stats()
                step()
                torch.cuda.synchronize()
                peak = torch.cuda.max_memory_allocated() - base
                ms = timed(step, 1, 3)
                res["N%d_%s_%s" % (N, mode, name)] = dict(ms_per_step=ms, peak_MB=peak / 1e6)
                log("%-7s forward_upsampled(k=250, image 256), general kernels, N=%3d %-13s %9.2f ms/step  peak %9.1f MB"
                    % (mode, N, name, ms, peak / 1e6))
        # 3. the synthesis launch alone against the fused debug launch
        L = _cabi.lib()
        V, M = 25, 2
        nbytes = int(L.vr_upsampled_workspace_bytes(N, T, V, M))
        work = torch.empty(nbytes // 8, dtype=torch.float64, device="cuda")
        iq = torch.empty(N, k * T, 2, device="cuda")
        out = torch.empty(N, 256, k * T // 16 + 1, device="cuda")
        stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        lay = frozen
        a = (x.data_ptr(), N, T, V, M, lay._src_c, lay._dst_c, len(lay.src), lay.wavelength.data_ptr(),
             lay.radar_location.data_ptr())

        def synth():
            _cabi.check(L.vr_synth_upsampled_f32(*a, 0, k, ctypes.c_float(3.0), work.data_ptr(), nbytes, iq.data_ptr(), stream))

        def debug():
            _cabi.check(L.vr_forward_upsampled_debug_f32(*a, 256, 16, 0, k, ctypes.c_float(3.0), work.data_ptr(), nbytes,
                                                         out.data_ptr(), iq.data_ptr(), stream))
        for name, fn in (("vr_synth_upsampled_f32", synth), ("vr_forward_upsampled_debug_f32", debug)):
            ms = timed(fn, 2, 10)
            res["N%d_%s" % (N, name)] = dict(ms=ms)
            log("kernel time N=%3d %-32s %9.3f ms" % (N, name, ms))
        del x, work, iq, out
    log(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
