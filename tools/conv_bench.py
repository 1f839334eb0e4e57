"""Direct convolution (conv2d_direct) against the im2col path (conv2d_im2col, workspace_images=16, AUTO and SIMT) on one GPU.

For each shape: warm-up, then CUDA-event timing of the arms in alternation (each round times every arm over `--iters`
back-to-back calls; the median round is reported), a bit-for-bit check of the direct output against im2col on PATH_SIMT
(and of the fused bias + ReLU against the same values put through x + bias, max(., 0)), and the algorithmic bytes and
FLOPs computed from the shapes, as fractions of the HBM bound (7.7 TB/s, the B200 data-sheet figure) and of the FP32 FFMA
bound (SMs x 128 FMA/clk x the SM clock nvidia-smi reports in the same run).  Prints a text table (and --out FILE).

    python tools/conv_bench.py [--iters 20] [--rounds 7] [--out FILE]"""
import argparse
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12
FMA_PER_CLK_PER_SM = 128

SHAPES = [   # name, ishape, kshape, padding, strides, fused bias + ReLU
    ("reference bench 16x3x224x224 -> 20x3x3", (16, 3, 224, 224), (20, 3, 3, 3), (0, 0), (1, 1), False),
    ("reference bench + bias + ReLU", (16, 3, 224, 224), (20, 3, 3, 3), (0, 0), (1, 1), True),
    ("ResNet stem 16x3x224x224 -> 64x7x7 s2 p3", (16, 3, 224, 224), (64, 3, 7, 7), (3, 3), (2, 2), False),
    ("large K 32x64x56x56 -> 64x3x3 p1", (32, 64, 56, 56), (64, 64, 3, 3), (1, 1), (1, 1), False),
]


def smi(fields):
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=" + fields, "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=60).stdout.strip().splitlines()
        return out[0] if out else "n/a"
    except (OSError, subprocess.SubprocessError):
        return "n/a"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import numpy as np
    import torch

    import laser_b200 as L

    assert torch.cuda.is_available(), "conv_bench needs a GPU"
    L.init()
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    props = torch.cuda.get_device_properties(0)
    sms = props.multi_processor_count
    say("device: %s | nvidia-smi name, power.limit, clocks.max.sm: %s" % (props.name, smi("name,power.limit,clocks.max.sm")))
    say("library: %s" % os.path.relpath(L.lib_path(), ROOT))
    say("timing: CUDA events, %d calls per round, median of %d rounds, arms alternating within each round" % (args.iters,
                                                                                                                 args.rounds))
    rows = []
    for name, ishape, kshape, padding, strides, fused in SHAPES:
        oshape = L.conv2d_out_shape(ishape, kshape, padding, strides)
        B, Cout = ishape[0], kshape[0]
        K = ishape[1] * kshape[2] * kshape[3]
        g = torch.Generator(device="cuda").manual_seed(7)
        tin = torch.rand(ishape, device="cuda", generator=g) * 2 - 1
        tker = torch.rand(kshape, device="cuda", generator=g) * 2 - 1
        bias = torch.rand((Cout,), device="cuda", generator=g) - 0.5 if fused else None
        out_d = torch.empty(oshape, device="cuda")
        out_a = torch.empty(oshape, device="cuda")
        out_s = torch.empty(oshape, device="cuda")
        per = L.im2col_workspace_size(ishape, kshape, padding, strides)
        wsi = min(16, B)
        ws = torch.empty(max(1, wsi * per), device="cuda")
        kw = dict(bias=bias, activation="relu") if fused else {}
        arms = {
            "direct": lambda: L.conv2d_direct(out_d, tin, ishape, tker, kshape, padding, strides, **kw),
            "im2col AUTO": lambda: L.conv2d_im2col(out_a, tin, ishape, tker, kshape, padding, strides, workspace=ws,
                                                   workspace_images=wsi, path=L.PATH_AUTO),
            "im2col SIMT": lambda: L.conv2d_im2col(out_s, tin, ishape, tker, kshape, padding, strides, workspace=ws,
                                                   workspace_images=wsi, path=L.PATH_SIMT),
        }
        for fn in arms.values():   # warm-up
            for _ in range(3):
                fn()
        torch.cuda.synchronize()
        times = {a: [] for a in arms}
        for _ in range(args.rounds):
            for a, fn in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.iters):
                    fn()
                e1.record()
                e1.synchronize()
                times[a].append(e0.elapsed_time(e1) / args.iters)
        clk = smi("clocks.sm")
        # bit identity with the exact im2col path (through x + bias, max(., 0) when fused)
        want = out_s if not fused else torch.clamp_min(out_s + bias.view(1, Cout, 1, 1), 0.0)
        same = torch.equal(out_d.view(torch.int32), want.view(torch.int32))
        nbytes = 4 * (int(np.prod(ishape)) + int(np.prod(kshape)) + int(np.prod(oshape)) + (Cout if fused else 0))
        flops = 2.0 * int(np.prod(oshape)) * K
        try:
            mhz = float(smi("clocks.max.sm").split()[0])
        except ValueError:
            mhz = float("nan")
        t_hbm = nbytes / HBM_BYTES_PER_S * 1e3
        t_ffma = flops / (2.0 * sms * FMA_PER_CLK_PER_SM * mhz * 1e6) * 1e3
        say()
        say("%s  (K = %d, c_out = %d, outputs %s)" % (name, K, Cout, "x".join(map(str, oshape))))
        say("  algorithmic bytes %.1f MB, FLOPs %.3f G; HBM bound %.4f ms, FFMA bound %.4f ms at %.0f MHz x %d SMs "
            "(the larger: %s); SM clock after timing: %s" % (nbytes / 1e6, flops / 1e9, t_hbm, t_ffma, mhz, sms,
                                                            "FFMA" if t_ffma > t_hbm else "HBM", clk))
        say("  direct output bit-identical to im2col SIMT%s: %s" % (" + bias + ReLU" if fused else "", same))
        for a in arms:
            ms = float(np.median(times[a]))
            say("  %-12s %8.4f ms   (min %.4f)  %5.1f %% of HBM bound, %5.1f %% of FFMA bound" % (
                a, ms, min(times[a]), 100 * t_hbm / ms, 100 * t_ffma / ms))
            rows.append((name, a, ms))
        del ws, out_d, out_a, out_s
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
