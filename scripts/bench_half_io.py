"""SpectralConv step with float32 / float16 / bfloat16 x on one GPU; prints ONE JSON line.

    python scripts/bench_half_io.py [--reps 60] [--warmup 10]

Per config (cfg-1 1024, cfg-2 128^2 headline, cfg-4 64^3, cfg-5 256^2): the fwd+bwd step of nb.SpectralConv replayed from a CUDA
graph, the three input dtypes alternating in one process (median of per-replay CUDA-event times; L2 overwritten with a 256 MB
buffer between timed replays, outside the events), the kernel times of one eager step from torch.profiler, the algorithmic bytes of
the step (x and dx at the input's width, y and gy fp32), the largest relative differences of y / dx against the float32 path, and the
reference's float16-autocast op sequence (cuFFT half transforms, complex-half contraction) on PyTorch as the denominator.  The card's
name and power limit are read in the same run."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import neuraloperator_b200 as nb  # noqa: E402
from neuraloperator_b200 import _lib  # noqa: E402

CONFIGS = [("cfg-2 FNO2d 128^2", 32, 64, (128, 128), (32, 32)), ("cfg-4 FNO3d 64^3", 8, 32, (64, 64, 64), (16, 16, 16)),
           ("cfg-5 FNO2d 256^2", 16, 64, (256, 256), (64, 64)), ("cfg-1 FNO1d 1024", 16, 32, (1024,), (16,))]
DTYPES = {"float32": torch.float32, "float16": torch.float16, "bfloat16": torch.bfloat16}


def step_bytes(B, Ci, Co, S, M, x_bytes):
    """x read + dx written at the input's width, y written + gy read in fp32, the weight (read twice + its gradient) and the
    kept-mode tensors (complex64) that cross HBM between the kernels.  For 16-bit input this is what the step moves where the fused
    tensor-core kernels read x / write dx directly; elsewhere the library adds an fp32 copy of x and of dx (two conversion launches
    per step, visible in `launches_per_step`), which these bytes do not count."""
    return 2 * x_bytes * B * Ci * S + 8 * B * Co * S + 24 * Ci * Co * M + 16 * B * Ci * M


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True,
                             timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return name, power
    except Exception as exc:  # noqa: BLE001
        return torch.cuda.get_device_name(0), f"unknown ({exc!r:.80})"


def capture(fn):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(3):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()
    return g


def timed_replays(graphs, warmup, reps, flush):
    """graphs: name -> graph; replayed alternately; returns name -> median ms."""
    times = {k: [] for k in graphs}
    for _ in range(warmup):
        for g in graphs.values():
            g.replay()
    torch.cuda.synchronize()
    for _ in range(reps):
        for k, g in graphs.items():
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            g.replay()
            e1.record()
            torch.cuda.synchronize()
            times[k].append(e0.elapsed_time(e1))
    return {k: statistics.median(v) for k, v in times.items()}


def profile_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t > 0:
            out[ev.key[:80]] = round(t / 1e3, 4)      # ms
    return out


def reference_autocast_step(conv, x16, gy, modes):
    """The reference's float16-autocast forward (rfftn in half, fftshift, kept block, einsum_complexhalf, complex64 spectrum, irfftn)
    and the backward autograd records for it."""
    d = len(modes)
    grid = tuple(x16.shape[2:])
    w = conv.weight.tensor.detach().clone().requires_grad_(True)
    bias = conv.bias.detach()
    dims = tuple(range(-d, 0))
    kept = [m for m in modes[:-1]] + [modes[-1] // 2 + 1]
    sl = [slice(None), slice(None)] + [slice(n // 2 - k // 2, n // 2 + k // 2) for n, k in zip(grid[:-1], kept[:-1])] + [slice(0, kept[-1])]
    letters = "xyzw"[:d]

    def fwd(x):
        xf = torch.fft.fftshift(torch.fft.rfftn(x, dim=dims, norm="forward"), dim=dims[:-1])
        xk = xf[tuple(sl)]
        xr, xi = xk.real, xk.imag
        wr, wi = w.real.half(), w.imag.half()
        eq = f"bi{letters},io{letters}->bo{letters}"
        yr = torch.einsum(eq, xr, wr) - torch.einsum(eq, xi, wi)
        yi = torch.einsum(eq, xr, wi) + torch.einsum(eq, xi, wr)
        out = torch.zeros(x.shape[0], w.shape[1], *grid[:-1], grid[-1] // 2 + 1, dtype=torch.complex64, device=x.device)
        out[tuple(sl)] = torch.complex(yr.float(), yi.float())
        out = torch.fft.ifftshift(out, dim=dims[:-1])
        return torch.fft.irfftn(out, s=grid, dim=dims, norm="forward") + bias

    xr = x16.detach().clone().requires_grad_(True)
    return lambda: torch.autograd.grad(fwd(xr), [xr, w], gy)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=60)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--configs", type=int, default=len(CONFIGS))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_half_io.py measures on the GPU; there is no CPU fallback"
    from bench import measured_peaks
    dev = torch.device("cuda", 0)
    name, power = card()
    peak, peak_src = measured_peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    result = {"card": name, "power_limit": power, "hbm_peak_gbs": peak, "hbm_peak_source": peak_src,
              "timing": f"CUDA graph replay, dtypes alternating, {args.warmup} warm-ups, median of {args.reps}, L2 overwritten between replays",
              "configs": {}}
    for cname, B, C, grid, modes in CONFIGS[:args.configs]:
        torch.manual_seed(0)
        conv = nb.SpectralConv(C, C, modes).to(dev)
        S = math.prod(grid)
        kept = list(modes[:-1]) + [modes[-1] // 2 + 1]
        M = math.prod(kept)
        x32 = torch.randn(B, C, *grid, device=dev)
        gy = torch.randn(B, C, *grid, device=dev)
        graphs, outs, kernels, launches = {}, {}, {}, {}
        params = list(conv.parameters())
        for dname, dt in DTYPES.items():
            x = x32.to(dt).requires_grad_(True)

            def step(x=x):
                # autograd.grad: fresh gradient buffers every step, no accumulation kernels in the timed graph
                return torch.autograd.grad(conv(x), [x, *params], gy)
            y = conv(x)
            dx = torch.autograd.grad(y, [x], gy)[0]
            torch.cuda.synchronize()
            outs[dname] = (y.detach(), dx)
            kernels[dname] = profile_kernels(step)
            c0 = _lib.launch_count()
            step()
            launches[dname] = _lib.launch_count() - c0
            graphs[dname] = capture(step)
        # the 16-bit runs against the float32 path on the same (widened) input
        errs = {}
        for dname, dt in DTYPES.items():
            if dt == torch.float32:
                continue
            xw = x32.to(dt).float().requires_grad_(True)
            yw = conv(xw)
            dxw = torch.autograd.grad(yw, [xw], gy)[0]
            yw = yw.detach()
            y16, dx16 = outs[dname]
            errs[dname] = {"y_max_rel_diff": ((y16 - yw).abs().max() / yw.abs().max()).item(),
                           "dx_max_rel_diff_vs_fp32_dx": ((dx16.float() - dxw).abs().max() / dxw.abs().max()).item(),
                           "dx_equals_fp32_dx_cast": bool(torch.equal(dx16, dxw.to(dt)))}
        ms = timed_replays(graphs, args.warmup, args.reps, flush)
        ref_ms = None
        if all(n & (n - 1) == 0 for n in grid):
            ref_step = reference_autocast_step(conv, x32.half(), gy, modes)
            ref_graph = capture(ref_step)
            ref_ms = timed_replays({"ref": ref_graph}, args.warmup, args.reps, flush)["ref"]
        entry = {"B": B, "C": C, "grid": list(grid), "modes": list(modes), "reference_fp16_autocast_ms": ref_ms, "dtypes": {},
                 "errors_vs_fp32_path": errs}
        for dname, dt in DTYPES.items():
            xb = torch.finfo(dt).bits // 8
            nbytes = step_bytes(B, C, C, S, M, xb)
            entry["dtypes"][dname] = {"step_ms": ms[dname], "algorithmic_bytes": nbytes,
                                      "hbm_frac": nbytes / (ms[dname] * 1e-3) / 1e9 / peak,
                                      "speedup_vs_reference": (ref_ms / ms[dname]) if ref_ms else None,
                                      "launches_per_step": launches[dname], "kernels_ms": kernels[dname]}
        result["configs"][cname] = entry
        del graphs
        torch.cuda.synchronize()
    print(json.dumps(result))


if __name__ == "__main__":
    main()
